"""The reference's evolutionary env classes — dict API over the CUDA step.

`PredPreyGrassEco`   ~ predpreygrass/evolutionary/eco_evolutionary/predpreygrass_rllib_env.py (ECO)
`PredPreyGrassStag`  ~ predpreygrass/evolutionary/stag_hunt_forward_view_nature_nurture/predpreygrass_rllib_env.py (STAG)

Same constructor (`config` dict with the reference's keys; ECO reads its mandatory keys with `config[...]`,
ECO:36-120, so a missing one raises KeyError here as well), same `reset(*, seed, options)` / `step(action_dict)`
returning agent-id string dicts with `"__all__"` (ECO:274-507, STAG:414-718), same spaces
(ECO:1396-1418, STAG:1784-1816) and the attributes the reference's `random_policy.py` / evaluation scripts read
(`agents`, `possible_agents`, `agent_positions`, `agent_energies`, `agent_ages`, `grass_positions`,
`grass_energies`, `agents_just_ate`, `current_step`, `active_num_predators/prey`, ECO `agent_genomes`-style speeds,
STAG `predator_facing`, `predator_cooperation_trait`, the team-capture counters).

One object = one env instance of a 1-env `BatchedPredPreyGrass` handle; all simulation work is done by the CUDA
kernels, this file converts the handle's row batch to the reference's dicts.  For throughput use
`BatchedPredPreyGrass` (thousands of envs, tensors stay on the GPU).

`reset(seed=s)` reproduces the reference's reset exactly: the numpy draws of the reference's reset
(ECO:130,208-215,1752 — founder speeds then `rng.choice` cells; STAG:273,2140-2169 — `rng.choice` cells, then per
founder predator a facing index and a raw cooperation trait) are made on the host from `np.random.default_rng(s)`
and handed to the device as a replay tape (`reference_reset_tape_eco` / `_stag`, pinned against the golden
recordings of the reference in tests/test_env_tapes.py).  Draws AFTER the reset (mutation, spawn fallback, capture
success) come from the device's Philox stream unless `options={"ppg_tape": (ints, reals)}` supplies the
reference's recorded draws (what the parity tests do).

Dict key order: ECO builds its return dicts from Python sets (ECO:413,424 — hash order, different in every
process), so this adapter uses (species, id) order.  STAG: live agents in `self.agents` order (STAG:551), then the
agents that ended this step sorted by id string (STAG:567-568).
"""
import numpy as np

from .config import (ENV_TERMINATED, ENV_TRUNCATED, ROW_ATE, ROW_FROZEN, ROW_REPRODUCED, ROW_TERMINATED, ROW_TRUNCATED, VARIANT_ECO,
                     VARIANT_STAG, make_config)
from .env import Box, Discrete, _Base, raise_on_status

try:
    from gymnasium.spaces import Dict as DictSpace
    from gymnasium.spaces import MultiDiscrete
except Exception:  # noqa: BLE001
    class MultiDiscrete:
        def __init__(self, nvec):
            self.nvec = np.asarray(nvec, np.int64)
            self.shape = self.nvec.shape
            self._rng = np.random.default_rng()

        def sample(self):
            return (self._rng.random(self.nvec.shape) * self.nvec).astype(np.int64)

        def contains(self, x):
            x = np.asarray(x)
            return x.shape == self.nvec.shape and bool((x >= 0).all() and (x < self.nvec).all())

    class DictSpace(dict):
        @property
        def spaces(self):
            return self

        def sample(self):
            return {k: v.sample() for k, v in self.items()}

FACING_OPTIONS = [(-1, -1), (-1, 0), (-1, 1), (0, -1), (0, 1), (1, -1), (1, 0), (1, 1)]  # STAG:197-206


# ---------------------------------------------------------------------------------------------- reset tapes
def reference_reset_tape_eco(seed, config):
    """The draws of ECO's `reset(seed)` in the tape layout of include/ppg.h: founders are registered first
    (one `rng.normal(mean, std)` each where std > 0, predators then prey; ECO:208-215, genome.py:31-36,42-46), then
    the cells come from one `rng.choice(G*G, n, replace=False)` (ECO:1752).  -> (cells int32, founder speeds f64)"""
    rng = np.random.default_rng(seed)
    G = config["grid_size"]
    n_pred, n_prey = config["n_initial_active_predators"], config["n_initial_active_prey"]
    speeds = []
    if config.get("genome_enabled", True):
        lo, hi = config.get("trait_bounds", {}).get("speed", (0.5, 2.0))
        for role, n in (("predator", n_pred), ("prey", n_prey)):
            f = config.get("founder_genome", {}).get(role, {})
            mean, std = f.get("speed_mean", 1.0), f.get("speed_std", 0.0)
            for _ in range(n):
                v = mean if std <= 0 else float(rng.normal(mean, std))
                speeds.append(float(np.clip(v, float(lo), float(hi))))
    cells = rng.choice(G * G, size=n_pred + n_prey + config["initial_num_grass"], replace=False)
    return np.asarray(cells, np.int32), np.asarray(speeds, np.float64)


def reference_reset_tape_stag(seed, config):
    """The draws of STAG's `reset(seed)`: `rng.choice(list(range(G*G)), n, replace=False)` (STAG:2140), then per
    founder predator `rng.integers(8)` (facing, STAG:941) and, with the cooperation trait enabled,
    `rng.normal(mean, std)` (STAG:1087).  -> (cells, facing indices, raw traits)"""
    g = config.get
    rng = np.random.default_rng(seed)
    G = config["grid_size"]
    n_pred = g("n_initial_active_type_1_predator", 0) + g("n_initial_active_type_2_predator", 0)
    n_prey = g("n_initial_active_type_1_prey", 0) + g("n_initial_active_type_2_prey", 0)
    walls = {(int(x), int(y)) for x, y in (g("manual_wall_positions") or []) if 0 <= x < G and 0 <= y < G}  # STAG:2107-2127
    free = [i for i in range(G * G) if (i // G, i % G) not in walls]  # STAG:2138
    cells = rng.choice(free, size=n_pred + n_prey + g("initial_num_grass", 0), replace=False)
    facing, traits = [], []
    for _ in range(n_pred):
        facing.append(int(rng.integers(8)))
        if g("coop_trait_enabled", True):
            # defaults of STAG:140-141 (the std is clamped at 0 there, as in config._fill_stag)
            traits.append(float(rng.normal(g("coop_trait_init_mean", 0.6), max(0.0, g("coop_trait_init_std", 0.12)))))
    return np.asarray(cells, np.int32), np.asarray(facing, np.int32), np.asarray(traits, np.float64)


# ---------------------------------------------------------------------------------------------- common adapter
class _RowDictEnv(_Base):
    """rows of env 0 of a 1-env handle  <->  the reference's per-agent dicts"""

    _variant = None
    _stay = 0
    _tolerated_status = 0  # status bits that are not an exception in the reference class mirrored

    def __init__(self, config=None):
        super().__init__()
        if config is None:
            raise ValueError("Environment config must be provided explicitly.")  # ECO:21-22, STAG:21-22
        from .batched import BatchedPredPreyGrass  # needs the CUDA extension; fails loudly without it

        self.config = config
        # STAG's visibility channel is a constant plane of ones in the reference (its line-of-sight masks are computed before
        # any wall exists, STAG:408-412): the device rows do not carry it, `_vis` appends it to the dict observations
        self._vis_plane = bool(self._variant == VARIANT_STAG and config.get("include_visibility_channel", False))
        if self._vis_plane:
            config = dict(config, include_visibility_channel=False)
        self._cfg = make_config(config, variant=self._variant, cap_live=config.get("cap_live"), autoreset=False,
                                seed=config.get("seed") or 0, track_episode_sums=self._variant == VARIANT_ECO)
        self._batch = BatchedPredPreyGrass(self._cfg, 1, device=config.get("cuda_device", 0))
        self.max_steps = config["max_steps"] if self._variant == VARIANT_ECO else config.get("max_steps", 0)  # ECO:43, STAG:127
        self.grid_size = self._cfg.grid_size
        self.num_obs_channels = self._cfg.num_obs_channels
        self.predator_obs_range, self.prey_obs_range = self._cfg.obs_range[0], self._cfg.obs_range[1]
        self.initial_num_grass = self._cfg.n_grass
        self.grass_agents = [f"grass_{k}" for k in range(self.initial_num_grass)]
        self.agents = []
        self.agents_just_ate = set()
        self.current_step = 0
        self._rows = {}
        self._done = True
        self._state = None

    # -- naming hooks
    def _name(self, s, i):
        raise NotImplementedError

    def _key(self, agent):
        raise NotImplementedError

    def _action(self, s, value):
        return int(value)

    def _read(self):
        raise NotImplementedError

    # -- reset / step plumbing
    def _reset_device(self, seed, cells, reals, options):
        b = self._batch
        extra = (options or {}).get("ppg_tape")
        if extra is not None:
            cells = np.concatenate([cells, np.asarray(extra[0], np.int32)])
            reals = np.concatenate([reals, np.asarray(extra[1], np.float64)])
        b.load_tape([cells], [reals])
        b.reset(seeds=np.array([np.uint64(int(seed) & 0xFFFFFFFFFFFFFFFF)], np.uint64))
        self.current_step = 0
        self._done = False
        self._state = None
        out = b.outputs_numpy()
        raise_on_status(int(out["env_status"][0]) & ~self._tolerated_status, self._variant)
        return out

    def _step_device(self, action_dict):
        import torch

        if self._done:
            raise RuntimeError("step() called on a finished episode; call reset()")
        self._state = None
        b = self._batch
        acts = [np.full(max(1, b.row_capacity[s]), self._stay, np.int32) for s in range(2)]
        order = [np.zeros(max(1, b.row_capacity[s]), np.int32) for s in range(2)]
        seen = [0, 0]
        for agent, action in action_dict.items():
            if agent not in self._rows:
                self._unknown_actor(agent)
                continue
            s, row = self._rows[agent]
            a = self._action(s, action)
            if not 0 <= (a & 0xFF) < self._n_moves(agent):
                raise KeyError(action)  # the reference indexes its action -> move table (ECO:668, STAG:834-841)
            acts[s][row] = a
            order[s][row] = seen[s]
            seen[s] += 1
        if seen[0] + seen[1] != len(self._rows):
            missing = [a for a in self._rows if a not in action_dict]
            raise KeyError(f"action_dict misses live agents {missing[:4]} (every live agent must act)")
        t = [torch.from_numpy(x).to(b.device) for x in acts + order]
        b.step_ordered(t[0], t[1], t[2], t[3])
        out = b.outputs_numpy()
        self.current_step = int(out["env_step"][0])
        raise_on_status(int(out["env_status"][0]) & ~self._tolerated_status, self._variant)
        return out

    def _n_moves(self, agent):
        raise NotImplementedError

    def _unknown_actor(self, agent):
        raise KeyError(agent)

    def _rows_of(self, out):
        """[(name, species, row, flags)] of env 0: rows of the agents that acted, then the newborn rows"""
        res = []
        for group in ("old", "new"):
            for s in range(2):
                if group == "old":
                    r0, r1 = int(out[f"old_off{s}"][0]), int(out[f"old_off{s}"][1])
                else:
                    r0 = int(out[f"new_off{s}"][0])
                    r1 = r0 + int(out[f"new_cnt{s}"][0])
                for r in range(r0, r1):
                    res.append((self._name(s, int(out[f"row_agent{s}"][r])), s, r, int(out[f"flags{s}"][r])))
        return res

    # -- attributes read by renderers / random_policy.py (ECO random_policy.py:75-82)
    @property
    def agent_positions(self):
        st = self._read()
        return {self._name(s, int(i)): (int(x), int(y)) for s in range(2) for i, (x, y) in zip(st["ids"][s], st["xy"][s])}

    @property
    def predator_positions(self):
        return {k: v for k, v in self.agent_positions.items() if "predator" in k}

    @property
    def prey_positions(self):
        return {k: v for k, v in self.agent_positions.items() if "prey" in k}

    @property
    def agent_energies(self):
        st = self._read()
        return {self._name(s, int(i)): float(e) for s in range(2) for i, e in zip(st["ids"][s], st["energy"][s])}

    @property
    def agent_ages(self):
        st = self._read()
        return {self._name(s, int(i)): int(a) for s in range(2) for i, a in zip(st["ids"][s], st["age"][s])}

    @property
    def grass_positions(self):
        st = self._read()
        return {f"grass_{k}": (int(x), int(y)) for k, (x, y) in enumerate(st["grass_xy"])}

    @property
    def grass_energies(self):
        st = self._read()
        return {f"grass_{k}": float(e) for k, e in enumerate(st["grass_energy"])}

    @property
    def grid_world_state(self):
        """the reference's `grid_world_state` (float32 [num_obs_channels, G, G], ECO / STAG / trait variants): the world
        after the last reset() / step().  After restore_state_snapshot() it is available again after the next step()."""
        return self._batch.world_state(0, 1)[0].cpu().numpy()

    def get_state_snapshot(self):
        return {"blob": self._batch.snapshot(), "current_step": self.current_step, "agents": list(self.agents),
                "agents_just_ate": set(self.agents_just_ate), "done": self._done}

    def restore_state_snapshot(self, snapshot):
        self._batch.restore(snapshot["blob"])
        self.current_step = snapshot["current_step"]
        self.agents = list(snapshot["agents"])
        self.agents_just_ate = set(snapshot["agents_just_ate"])
        self._done = snapshot["done"]
        self._state = None
        out = self._batch.outputs_numpy()  # ppg_restore relabels the rows densely in list order
        self._rows = {}
        for s in range(2):
            off = out[f"old_off{s}"]
            for r in range(int(off[0]), int(off[1])):
                self._rows[self._name(s, int(out[f"row_agent{s}"][r]))] = (s, r)

    def close(self):
        if getattr(self, "_batch", None) is not None:
            self._batch.close()
            self._batch = None


# ---------------------------------------------------------------------------------------------- ECO
class PredPreyGrassEco(_RowDictEnv):
    """eco_evolutionary `PredPreyGrass(config)`: heritable speed trait, 25 actions, move cost, ageing, carcasses."""

    _variant = VARIANT_ECO
    _events_supported = True  # per_step_agent_data / agent_event_log (event_log.py) follow eco_evolutionary's energy rules

    def __init__(self, config=None):
        super().__init__(config)
        c = self._cfg
        self.n_possible_predators, self.n_possible_prey = config["n_possible_predators"], config["n_possible_prey"]
        self.n_initial_active_predators, self.n_initial_active_prey = c.n_initial[0], c.n_initial[1]
        self.action_range = config["action_range"]
        self.genome_enabled = bool(c.genome_enabled)
        self.include_speed_in_obs = bool(c.include_speed_in_obs)
        self.speed_distance_threshold = c.speed_distance_threshold
        self._stay = (self.action_range * self.action_range) // 2
        self.possible_agents = [f"predator_{i}" for i in range(self.n_possible_predators)] + [
            f"prey_{j}" for j in range(self.n_possible_prey)]  # ECO:1378-1394
        C = self.num_obs_channels + (1 if self.include_speed_in_obs else 0)  # ECO:1396-1406
        pred_space = Box(low=0, high=100.0, shape=(C, self.predator_obs_range, self.predator_obs_range), dtype=np.float32)
        prey_space = Box(low=0, high=100.0, shape=(C, self.prey_obs_range, self.prey_obs_range), dtype=np.float32)
        act = Discrete(self.action_range ** 2)
        self.observation_spaces = {a: pred_space if "predator" in a else prey_space for a in self.possible_agents}
        self.action_spaces = {a: act for a in self.possible_agents}
        self.observation_space = DictSpace(self.observation_spaces)
        self.action_space = DictSpace(self.action_spaces)
        d = (self.action_range - 1) // 2  # ECO:225-232
        self.action_to_move_tuple_agents = {i: (i // self.action_range - d, i % self.action_range - d) for i in range(self.action_range ** 2)}
        # the exporters of the evaluation scripts (ECO:426-446, 1575-1597); "record_agent_events": False switches them off
        # (they cost one read-back of the env's agent lists per step)
        self._events = None
        if self._events_supported and config.get("record_agent_events", True):
            from .event_log import EcoEventRecorder

            self._events = EcoEventRecorder(config, self.action_to_move_tuple_agents, self.grid_size, self.speed_distance_threshold)

    def _name(self, s, i):
        return f"predator_{i}" if s == 0 else f"prey_{i}"

    def _event_state(self):
        """{agent: (position, energy, age, genome speed or None, member of dead_prey)} and {cell: (grass id, energy)} of the env"""
        st = self._read()
        state = {}
        for s in range(2):
            for k, i in enumerate(st["ids"][s]):
                state[self._name(s, int(i))] = ((int(st["xy"][s][k][0]), int(st["xy"][s][k][1])), float(st["energy"][s][k]), int(st["age"][s][k]),
                                                float(st["speed"][s][k]) if self.genome_enabled else None,
                                                bool(st["dead_prey"][k]) if s == 1 else False)
        grass = {(int(x), int(y)): (f"grass_{k}", float(e)) for k, ((x, y), e) in enumerate(zip(st["grass_xy"], st["grass_energy"]))}
        return state, grass

    # the reference's attributes (ECO:161-170), read by evaluate_ppo_from_checkpoint_*.py and the renderer's tooltips
    @property
    def per_step_agent_data(self):
        return self._events.per_step_agent_data if self._events else []

    @property
    def agent_event_log(self):
        return self._events.agent_event_log if self._events else {}

    @property
    def agent_parents(self):
        return self._events.agent_parents if self._events else {}

    @property
    def agent_offspring_counts(self):
        return self._events.agent_offspring_counts if self._events else {}

    @property
    def agent_live_offspring_ids(self):
        return self._events.agent_live_offspring_ids if self._events else {}

    def get_state_snapshot(self):
        """ECO:1277-1330: the snapshot carries the exporters' state as well"""
        import copy

        snap = super().get_state_snapshot()
        snap["events"] = copy.deepcopy(self._events)
        snap["episode_speeds"] = copy.deepcopy(getattr(self, "_episode_speeds", None))
        return snap

    def restore_state_snapshot(self, snapshot):
        import copy

        super().restore_state_snapshot(snapshot)
        if "events" in snapshot:
            self._events = copy.deepcopy(snapshot["events"])
        if snapshot.get("episode_speeds") is not None:
            self._episode_speeds = copy.deepcopy(snapshot["episode_speeds"])

    def get_all_agent_stats(self):
        """ECO:1676-1682: copies of all agent records (`agent_stats_live` then `agent_stats_completed`), rebuilt by the event recorder"""
        if self._events is None or not hasattr(self._events, "get_all_agent_stats"):
            raise RuntimeError("agent records are kept by the event recorder (record_agent_events=False)")
        return self._events.get_all_agent_stats()

    def get_total_offspring_by_type(self):
        """ECO:1705-1712"""
        if self._events is None or not hasattr(self._events, "get_total_offspring_by_type"):
            raise RuntimeError("agent records are kept by the event recorder (record_agent_events=False)")
        return self._events.get_total_offspring_by_type()

    def get_total_energy_by_type(self):
        """ECO:1684-1703: total energy of the live predators, the live prey and the grass"""
        st = self._read()
        totals = {"predator": 0.0, "prey": 0.0, "grass": sum(float(e) for e in st["grass_energy"])}
        for s, role in enumerate(("predator", "prey")):
            for e in st["energy"][s]:
                totals[role] += float(e)
        return totals

    def export_agent_event_log(self, path):
        """ECO:1575-1597"""
        if self._events is None:
            raise RuntimeError("agent events are not recorded (record_agent_events=False, or a trait variant)")
        self._events.export(path)

    def _n_moves(self, agent):
        return self.action_range ** 2

    def _read(self):
        if self._state is None:
            self._state = self._batch.read_env_eco(0)
        return self._state

    def reset(self, *, seed=None, options=None):
        super().reset(seed=seed)
        if seed is None:
            seed = self.config["seed"]  # ECO:128-129
        cells, speeds = reference_reset_tape_eco(seed, self.config)
        out = self._reset_device(seed, cells, speeds, options)
        obs, *_ = self._dicts(out)
        self.agents = list(obs)
        # genome speeds of every agent of the episode, founders first (the records `_build_episode_training_metrics` walks)
        self._episode_speeds = ([], [])
        if self.genome_enabled:
            st = self._read()
            for s in range(2):
                self._episode_speeds[s].extend(float(v) for v in st["speed"][s])
        if self._events is not None:
            state, grass = self._event_state()
            self._events.reset(state, self.agents, grass)
        return obs, {}

    def _dicts(self, out):
        obs, rew, term, trunc = {}, {}, {}, {}
        self._rows, self.agents_just_ate = {}, set()
        rows = sorted(self._rows_of(out), key=lambda t: (t[1], int(t[0].rsplit("_", 1)[1])))
        for name, s, r, f in rows:
            obs[name] = out[f"obs{s}"][r]
            rew[name] = float(out[f"reward{s}"][r])
            term[name] = bool(f & ROW_TERMINATED)
            trunc[name] = bool(f & ROW_TRUNCATED)
            if f & ROW_ATE:
                self.agents_just_ate.add(name)
            if not f & (ROW_TERMINATED | ROW_TRUNCATED):
                self._rows[name] = (s, r)
        return obs, rew, term, trunc

    def step(self, action_dict):
        t = self.current_step
        out = self._step_device(action_dict)
        obs, rew, term, trunc = self._dicts(out)
        flags = int(out["env_flags"][0])
        if self._events is not None:
            rows = self._rows_of(out)
            n_old = sum(int(out[f"old_off{s}"][1]) - int(out[f"old_off{s}"][0]) for s in range(2))
            newborn = sorted((name for name, s, r, f in rows[n_old:]), key=lambda a: ("prey" in a, int(a.rsplit("_", 1)[1])))
            state, grass = self._event_state()
            self._events.step(t, action_dict, {name: f for name, s, r, f in rows}, state, newborn, grass, bool(flags & ENV_TRUNCATED))
        if self.genome_enabled and (int(out["new_cnt0"][0]) or int(out["new_cnt1"][0])):
            st = self._read()  # newborns join the episode's agent records with their (mutated) genome
            by_id = [dict(zip(st["ids"][s].tolist(), st["speed"][s].tolist())) for s in range(2)]
            for s in range(2):
                r0 = int(out[f"new_off{s}"][0])
                for r in range(r0, r0 + int(out[f"new_cnt{s}"][0])):
                    self._episode_speeds[s].append(float(by_id[s][int(out[f"row_agent{s}"][r])]))
        infos = {a: {} for a in rew}
        term["__all__"] = bool(flags & ENV_TERMINATED)   # ECO:392,408 extinction
        trunc["__all__"] = bool(flags & ENV_TRUNCATED)   # ECO:452-486 time limit, same call
        if flags & (ENV_TERMINATED | ENV_TRUNCATED):
            self._done = True
            self.agents = []  # ECO:495,500-501
            self._rows = {}
            infos["__all__"] = {"training_metrics": self.episode_training_metrics()}  # ECO:1663-1668, 485
        else:
            # `self.agents` keeps insertion order: survivors, then this step's newborns, predators first (ECO:353-367)
            prev = set(self.agents)
            self.agents = [a for a in self.agents if a in self._rows] + [a for a in self._rows if a not in prev]
        return obs, rew, term, trunc, infos

    # ECO attributes
    @property
    def active_num_predators(self):
        return int(self._read()["active_num"][0])

    @property
    def active_num_prey(self):
        return int(self._read()["active_num"][1])

    @property
    def agent_speeds(self):
        """`{agent: agent_genomes[agent].speed}` (ECO:168,575-580)"""
        st = self._read()
        return {self._name(s, int(i)): float(v) for s in range(2) for i, v in zip(st["ids"][s], st["speed"][s])}

    @property
    def dead_prey(self):
        st = self._read()
        return {self._name(1, int(i)) for i, d in zip(st["ids"][1], st["dead_prey"]) if d}

    def episode_training_metrics(self):
        """`_build_episode_training_metrics` (ECO:1613-1661), same keys: over ALL agent records of the episode (alive or
        not) the speed distribution, and the per-agent means of distance travelled, locomotion energy spent and offspring
        count.  The totals come from the device (ppg_read_episode_eco); a mean over records is total / record count."""
        ep = self._batch.read_episode_eco(0)
        res = {}
        thr = float(self.speed_distance_threshold)
        for s, role in enumerate(("predator", "prey")):
            v = np.asarray(self._episode_speeds[s], np.float64)
            if v.size:
                p25, p50, p75 = np.percentile(v, [25, 50, 75])
                vals = (float(np.mean(v)), float(np.std(v)), float(p25), float(p50), float(p75), float(np.mean(v >= thr)))
            else:
                vals = (0.0,) * 6
            for key, x in zip(("speed_mean", "speed_std", "speed_p25", "speed_p50", "speed_p75", "fraction_fast"), vals):
                res[f"{role}_{key}"] = x
            count = int(self._cfg.n_initial[s]) + ep["spawned"][s]
            if count:
                res[f"{role}_distance_traveled_mean"] = ep["distance"][s] / count
                res[f"{role}_movement_energy_spent_mean"] = ep["move_energy"][s] / count
                res[f"{role}_offspring_count_mean"] = ep["spawned"][s] / count
                res[f"{role}_agent_count"] = float(count)
            else:
                for key in ("distance_traveled_mean", "movement_energy_spent_mean", "offspring_count_mean", "agent_count"):
                    res[f"{role}_{key}"] = 0.0
        return res

    def live_speed_metrics(self):
        """`_build_live_speed_metrics` (ECO:509-539): speed distribution of the live population, same keys"""
        st = self._read()
        res = {}
        for s, role in enumerate(("predator", "prey")):
            v = np.asarray(st["speed"][s], np.float64) if self.genome_enabled else np.zeros(0)
            if v.size:
                p25, p50, p75 = np.percentile(v, [25, 50, 75])
                vals = (float(v.mean()), float(v.std()), float(p25), float(p50), float(p75),
                        float((v >= float(self.speed_distance_threshold)).mean()), float(v.size))
            else:
                vals = (0.0,) * 7
            for key, x in zip(("speed_mean", "speed_std", "speed_p25", "speed_p50", "speed_p75", "fraction_fast", "count"), vals):
                res[f"{role}_{key}"] = x
        return res


# ---------------------------------------------------------------------------------------------- other heritable traits
def reference_reset_tape_trait(seed, config, trait):
    """The draws of the trait variants' `reset(seed)` in the tape layout of include/ppg.h (MR:189-200, genome.py
    `founder_genome`, MR:1469-1473): `rng.integers(min, max + 1)` for the number of predators, then of prey; one
    `rng.normal(mean, std)` per founder where std > 0 (predators then prey), clipped to the trait bounds; then one
    `rng.choice(G*G, n, replace=False)` for the cells.  -> (ints = [n_pred, n_prey, cells...], founder trait values)"""
    from .config import TRAIT_DEFAULTS

    rng = np.random.default_rng(seed)
    G = config["grid_size"]
    n_max = (config["n_initial_active_predators"], config["n_initial_active_prey"])
    n_min = (min(int(config.get("n_initial_active_predators_min", max(1, n_max[0] // 3))), n_max[0]),
             min(int(config.get("n_initial_active_prey_min", max(1, n_max[1] // 3))), n_max[1]))
    n = [int(rng.integers(n_min[s], n_max[s] + 1)) for s in range(2)]
    values = []
    if config.get("genome_enabled", True):
        default_mean, default_bounds = TRAIT_DEFAULTS[trait]
        lo, hi = config.get("trait_bounds", {}).get(trait, default_bounds)
        for role, k in (("predator", n[0]), ("prey", n[1])):
            f = config.get("founder_genome", {}).get(role, {})
            mean, std = f.get(f"{trait}_mean", default_mean), f.get(f"{trait}_std", 0.0)
            for _ in range(k):
                v = mean if std <= 0 else float(rng.normal(mean, std))
                values.append(float(np.clip(v, float(lo), float(hi))))
    cells = rng.choice(G * G, size=n[0] + n[1] + config["initial_num_grass"], replace=False)
    return np.concatenate([np.asarray(n, np.int32), np.asarray(cells, np.int32)]), np.asarray(values, np.float64)


class _TraitEnv(PredPreyGrassEco):
    """Shared dict adapter of the trait variants of eco_evolutionary (MR / INV / COOP): 9 actions, 3-channel windows, a
    random number of founders per episode, ids never reused, `infos["__all__"]["training_metrics"]` at the episode's end."""

    _trait = None
    _events_supported = False  # the trait variants' energy rules differ (rates, investment, meal sharing): no event recorder
    _tolerated_status = 0x10  # PPG_STATUS_ID_POOL_EMPTY: the trait variants print a warning and skip the birth (MR:856-864)
    _tag = None  # prefix of the reproduction-correlation keys (MR:1370-1392, COOP:1396-1418)

    def __init__(self, config=None):
        if config is None:
            raise ValueError("Environment config must be provided explicitly.")
        config = dict(config, ppg_trait=self._trait)
        super().__init__(config)
        self.n_initial_active_predators_min, self.n_initial_active_prey_min = self._cfg.n_initial_min[0], self._cfg.n_initial_min[1]
        self._records = ({}, {})
        # per_step_agent_data / agent_event_log (MR:391-411, 1153-1165) for the variants whose energy chain the recorder follows
        if config.get("record_agent_events", True):
            from .event_log import TraitEventRecorder

            self._events = TraitEventRecorder(config, self.action_to_move_tuple_agents, self.grid_size, self._trait)

    def reset(self, *, seed=None, options=None):
        _Base.reset(self, seed=seed)
        if seed is None:
            seed = self.config["seed"]  # MR:120-121
        ints, values = reference_reset_tape_trait(seed, self.config, self._trait)
        out = self._reset_device(seed, ints, values, options)
        obs, *_ = self._dicts(out)
        self.agents = list(obs)
        st = self._read()
        # one record per agent of the episode (`_iter_all_agent_records`, MR:1397-1404): trait value, offspring, energies
        self._records = ({}, {})
        for s in range(2):
            for i, v in zip(st["ids"][s].tolist(), st["speed"][s].tolist()):
                self._records[s][i] = self._new_record(v)
        self.peak_active_predators = self.peak_active_prey = 0  # MR:177-178
        if self._events is not None:
            state, grass = self._event_state()
            self._events.reset(state, self.agents, grass)
        return obs, {}

    @staticmethod
    def _new_record(trait_value, initial_energy=0.0):
        return {"trait": float(trait_value), "offspring": 0, "initial_energy": float(initial_energy), "invested": [], "after": []}

    def step(self, action_dict):
        t = self.current_step
        out = self._step_device(action_dict)
        obs, rew, term, trunc = self._dicts(out)
        flags = int(out["env_flags"][0])
        if self._events is not None:
            rows = self._rows_of(out)
            n_old = sum(int(out[f"old_off{s}"][1]) - int(out[f"old_off{s}"][0]) for s in range(2))
            newborn = sorted((name for name, s, r, f in rows[n_old:]), key=lambda a: ("prey" in a, int(a.rsplit("_", 1)[1])))
            state, grass = self._event_state()
            self._events.step(t, action_dict, {name: f for name, s, r, f in rows}, state, newborn, grass, bool(flags & ENV_TRUNCATED))
        if int(out["new_cnt0"][0]) or int(out["new_cnt1"][0]):
            # births run in predator_positions / prey_positions order (MR:318-331) = the order of the acting rows, and the
            # newborn rows are in birth order: the k-th parent flagged PPG_ROW_REPRODUCED is the parent of the k-th newborn
            st = self._read()
            for s in range(2):
                e_of = dict(zip(st["ids"][s].tolist(), st["energy"][s].tolist()))
                t_of = dict(zip(st["ids"][s].tolist(), st["speed"][s].tolist()))
                parents = [int(out[f"row_agent{s}"][r]) for r in range(int(out[f"old_off{s}"][0]), int(out[f"old_off{s}"][1]))
                           if int(out[f"flags{s}"][r]) & ROW_REPRODUCED]
                r0 = int(out[f"new_off{s}"][0])
                kids = [int(out[f"row_agent{s}"][r]) for r in range(r0, r0 + int(out[f"new_cnt{s}"][0]))]
                for par, kid in zip(parents, kids):
                    ce = float(e_of.get(kid, self._cfg.initial_energy[s]))
                    self._records[s][kid] = self._new_record(t_of.get(kid, -1.0), ce)  # MR:908 offspring_initial_energy
                    rec = self._records[s][par]
                    rec["offspring"] += 1
                    rec["invested"].append(ce)                       # MR:902-903
                    if par in e_of:
                        rec["after"].append(float(e_of[par]))        # MR:904-905 (reproduction is the step's last phase)
        infos = {a: {} for a in rew}
        term["__all__"] = bool(flags & ENV_TERMINATED)   # MR:354-374 extinction
        trunc["__all__"] = bool(flags & ENV_TRUNCATED)   # MR:418-461 time limit
        if flags & (ENV_TERMINATED | ENV_TRUNCATED):
            self._done = True
            self.agents = []
            self._rows = {}
            infos["__all__"] = {"training_metrics": self.episode_training_metrics()}  # MR:1394-1396, 458
        else:
            prev = set(self.agents)
            self.agents = [a for a in self.agents if a in self._rows] + [a for a in self._rows if a not in prev]
            n_pred = sum(1 for a in self.agents if "predator" in a)  # MR:466-471
            self.peak_active_predators = max(self.peak_active_predators, n_pred)
            self.peak_active_prey = max(self.peak_active_prey, len(self.agents) - n_pred)
        return obs, rew, term, trunc, infos

    @property
    def agent_traits(self):
        """`{agent: getattr(agent_genomes[agent], <trait>)}`"""
        return self.agent_speeds

    def episode_training_metrics(self):
        """`_build_episode_training_metrics` of the trait variants (MR:1274-1392): the trait distribution and the per-agent
        means over ALL agent records of the episode, spawn / peak / id counters and (MR, COOP) the reproduction rate per
        trait quartile.  Distance and locomotion totals and the event counters (births blocked by the id pool or the density
        cap, catches blocked by satiation, COOP's donated energy) come from the device (ppg_read_episode_eco,
        ppg_read_episode_events_eco); the `*_repro_spearman` rank correlations and COOP's `*_local_relatedness_proxy` come from
        the event recorder (the order of the agent records, the parents) and are left out with `record_agent_events: False`."""
        ep = self._batch.read_episode_eco(0)
        ev = self._batch.read_episode_events_eco(0)
        res, t = {}, self._trait
        for s, role in enumerate(("predator", "prey")):
            recs = list(self._records[s].values())
            v = np.asarray([r["trait"] for r in recs if self.genome_enabled], np.float64)
            if v.size:
                p25, p50, p75 = np.percentile(v, [25, 50, 75])
                vals = (float(np.mean(v)), float(np.std(v)), float(p25), float(p50), float(p75))
            else:
                vals = (0.0,) * 5
            for key, x in zip(("mean", "std", "p25", "p50", "p75"), vals):
                res[f"{role}_{t}_{key}"] = x
            if recs:
                n = len(recs)
                res[f"{role}_distance_traveled_mean"] = ep["distance"][s] / n
                res[f"{role}_movement_energy_spent_mean"] = ep["move_energy"][s] / n
                res[f"{role}_offspring_count_mean"] = float(np.mean([float(r["offspring"]) for r in recs]))
                res[f"{role}_agent_count"] = float(n)
                res[f"{role}_offspring_initial_energy_mean"] = float(np.mean([r["initial_energy"] for r in recs]))
                inv = [sum(r["invested"]) / len(r["invested"]) for r in recs if r["invested"]]
                aft = [sum(r["after"]) / len(r["after"]) for r in recs if r["after"]]
                res[f"{role}_reproduction_energy_invested_mean"] = float(np.mean(inv)) if inv else 0.0
                res[f"{role}_parent_energy_after_reproduction_mean"] = float(np.mean(aft)) if aft else 0.0
                if t == "cooperation_rate":  # COOP:1349-1354: every donated unit is received by the same species (COOP:585-586)
                    res[f"{role}_energy_donated_mean"] = ev["donated"][s] / n
                    res[f"{role}_energy_received_mean"] = ev["donated"][s] / n
            else:
                for key in ("distance_traveled_mean", "movement_energy_spent_mean", "offspring_count_mean", "agent_count",
                            "offspring_initial_energy_mean", "reproduction_energy_invested_mean", "parent_energy_after_reproduction_mean"):
                    res[f"{role}_{key}"] = 0.0
                if t == "cooperation_rate":
                    res[f"{role}_energy_donated_mean"] = res[f"{role}_energy_received_mean"] = 0.0
        if t == "cooperation_rate":  # COOP:1365-1368
            for s, role in enumerate(("predator", "prey")):
                res[f"{role}_energy_donated_total"] = res[f"{role}_energy_received_total"] = ev["donated"][s]
                if self._events is not None:  # kinship needs the parents, which the event recorder keeps (COOP:529-535, 1369-1371)
                    donated = self._events.energy_donated[s]
                    res[f"{role}_local_relatedness_proxy"] = float(self._events.kin_donation[s] / donated) if donated > 0.0 else 0.0
        res["predator_reproduction_blocked"] = float(ev["blocked_capacity"][0])  # MR:1347-1350
        res["prey_reproduction_blocked"] = float(ev["blocked_capacity"][1])
        if t == "metabolic_rate":
            res["predator_reproduction_blocked_density"] = float(ev["blocked_density"])
        if t in ("metabolic_rate", "offspring_investment_fraction"):
            res["predator_satiation_blocked_catches"] = float(ev["satiation_blocked"])
        res["predator_spawned_total"] = float(ep["spawned"][0])
        res["prey_spawned_total"] = float(ep["spawned"][1])
        res["peak_active_predators"] = float(self.peak_active_predators)
        res["peak_active_prey"] = float(self.peak_active_prey)
        res["prey_unique_ids_used"] = float(len(self._records[1]))
        res["predator_unique_ids_used"] = float(len(self._records[0]))
        if self._tag and self.genome_enabled:
            for s, role in ((1, "prey"), (0, "predator")):
                recs = list(self._records[s].values())
                if len(recs) < 4:
                    continue
                if self._events is not None:
                    # `{role}_{tag}_repro_spearman` (MR:1358-1382): the reference ranks with argsort and no tie correction, so the
                    # value depends on the order its record dicts are iterated in — live records, then the completed ones in
                    # the order they were closed, which the event recorder keeps
                    ids = [int(a.rsplit("_", 1)[1]) for a in self._events.record_order() if a.startswith(role)]
                    recs = [self._records[s][i] for i in ids]
                x = np.array([r["trait"] for r in recs])
                y = np.array([float(r["offspring"] > 0) for r in recs])
                if self._events is not None:
                    rx, ry = np.argsort(np.argsort(x)).astype(float), np.argsort(np.argsort(y)).astype(float)
                    rx -= rx.mean()
                    ry -= ry.mean()
                    denom = np.sqrt((rx ** 2).sum() * (ry ** 2).sum())
                    res[f"{role}_{self._tag}_repro_spearman"] = float(np.dot(rx, ry) / denom) if denom > 0.0 else 0.0
                q25, q50, q75 = np.percentile(x, [25, 50, 75])
                for k, m in enumerate((x <= q25, (x > q25) & (x <= q50), (x > q50) & (x <= q75), x > q75), 1):
                    if m.sum() > 0:
                        res[f"{role}_{self._tag}_repro_rate_q{k}"] = float(y[m].mean())
        return res

    def live_genome_metrics(self):
        """`_build_live_genome_metrics` (MR:476-504): trait distribution of the live population, same keys"""
        st = self._read()
        res, t = {}, self._trait
        for s, role in enumerate(("predator", "prey")):
            v = np.asarray(st["speed"][s], np.float64) if self.genome_enabled else np.zeros(0)
            if v.size:
                p25, p50, p75 = np.percentile(v, [25, 50, 75])
                vals = (float(v.mean()), float(v.std()), float(p25), float(p50), float(p75), float(v.size))
            else:
                vals = (0.0,) * 6
            for key, x in zip((f"{t}_mean", f"{t}_std", f"{t}_p25", f"{t}_p50", f"{t}_p75", "count"), vals):
                res[f"{role}_{key}"] = x
        return res


class PredPreyGrassMetabolicRate(_TraitEnv):
    """eco_evolutionary_metabolic_rate `PredPreyGrass(config)`: heritable metabolic rate (basal cost x rate, gains x rate ** alpha)."""

    _trait, _tag = "metabolic_rate", "mr"


class PredPreyGrassInvestment(_TraitEnv):
    """eco_evolutionary_investment `PredPreyGrass(config)`: heritable offspring investment fraction (child energy = parent's x fraction)."""

    _trait, _tag = "offspring_investment_fraction", None


class PredPreyGrassCooperation(_TraitEnv):
    """eco_evolutionary_cooperation `PredPreyGrass(config)`: heritable cooperation rate (a share of every meal goes to neighbours)."""

    _trait, _tag = "cooperation_rate", "coop"


# ---------------------------------------------------------------------------------------------- cadence
def reference_reset_tape_cadence(seed, config):
    """The draws of the cadence variant's `reset(seed)` in the tape layout of include/ppg.h: per founder (predators, then prey)
    `rng.normal(mean, std)` where std > 0 (genome.py founder_genome, clipped to the trait bounds) and then
    `rng.uniform(0.0, 1.0)` for the move accumulator (CAD:1324-1327); then one `rng.choice(G*G, n, replace=False)` for the cells.
    -> (cells int32, [speeds..., accumulators...] f64: the device reads all speeds first)"""
    rng = np.random.default_rng(seed)
    G = config["grid_size"]
    n = (config["n_initial_active_predators"], config["n_initial_active_prey"])
    genome = config.get("genome_enabled", True)
    lo, hi = config.get("trait_bounds", {}).get("speed", (0.5, 2.0))
    speeds, accs = [], []
    for role, k in (("predator", n[0]), ("prey", n[1])):
        f = config.get("founder_genome", {}).get(role, {})
        mean, std = f.get("speed_mean", 1.0), f.get("speed_std", 0.0)
        for _ in range(k):
            if genome:
                v = mean if std <= 0 else float(rng.normal(mean, std))
                speeds.append(float(np.clip(v, float(lo), float(hi))))
            accs.append(float(rng.uniform(0.0, 1.0)))
    cells = rng.choice(G * G, size=n[0] + n[1] + config["initial_num_grass"], replace=False)
    return np.asarray(cells, np.int32), np.asarray(speeds + accs, np.float64)


class PredPreyGrassCadence(PredPreyGrassEco):
    """eco_evolutionary_cadence `PredPreyGrass(config)`: the speed genome sets how OFTEN an agent may move (a per-agent
    accumulator, CAD:556-585,674-681); observations are dicts {"observations": window, "action_mask": 9 floats} whose mask
    allows only "stay" on the steps the agent will be frozen (device row flag PPG_ROW_FROZEN)."""

    _tolerated_status = 0
    _events_supported = False

    def __init__(self, config=None):
        if config is None:
            raise ValueError("Environment config must be provided explicitly.")
        config = dict(config, ppg_trait="cadence", lineage_reward_coeff=0.0)
        super().__init__(config)
        self.max_cooldown = int(config.get("max_cooldown", 10))
        n_act = self.action_range ** 2
        self._stay_action_index = n_act // 2
        mask_space = Box(low=0.0, high=1.0, shape=(n_act,), dtype=np.float32)
        C = self.num_obs_channels + (1 if self.include_speed_in_obs else 0)  # CAD:1277-1296: spatial Box(-100, 100) + mask
        sp = {0: Box(low=-100.0, high=100.0, shape=(C, self.predator_obs_range, self.predator_obs_range), dtype=np.float32),
              1: Box(low=-100.0, high=100.0, shape=(C, self.prey_obs_range, self.prey_obs_range), dtype=np.float32)}
        self.observation_spaces = {a: DictSpace({"observations": sp[0 if "predator" in a else 1], "action_mask": mask_space})
                                   for a in self.possible_agents}
        self.observation_space = DictSpace(self.observation_spaces)
        self._all = np.ones(n_act, np.float32)
        self._stay_only = np.zeros(n_act, np.float32)
        self._stay_only[self._stay_action_index] = 1.0
        if config.get("record_agent_events", True):  # agent_event_log, and per_step_agent_data with "record_step_data" (CAD:83,422)
            from .event_log import TraitEventRecorder

            self._events = TraitEventRecorder(config, self.action_to_move_tuple_agents, self.grid_size, "speed")

    def _event_state(self):
        """as the base class's, with the move accumulator (CAD:183-186) in the last place"""
        state, grass = super()._event_state()
        acc = self.agent_move_accumulator
        return {a: v[:4] + (acc[a],) for a, v in state.items()}, grass

    def _mask_dicts(self, out, obs):
        """window + row flag -> the reference's observation dict (CAD:746-753)"""
        flags = {self._name(s, int(out[f"row_agent{s}"][r])): int(out[f"flags{s}"][r]) for _, s, r, _ in self._rows_of(out)}
        return {a: {"observations": o, "action_mask": (self._stay_only if flags[a] & ROW_FROZEN else self._all).copy()} for a, o in obs.items()}

    def reset(self, *, seed=None, options=None):
        _Base.reset(self, seed=seed)
        if seed is None:
            seed = self.config["seed"]
        cells, reals = reference_reset_tape_cadence(seed, self.config)
        out = self._reset_device(seed, cells, reals, options)
        obs, *_ = self._dicts(out)
        self.agents = list(obs)
        self._episode_speeds = ([], [])
        if self.genome_enabled:
            st = self._read()
            for s in range(2):
                self._episode_speeds[s].extend(float(v) for v in st["speed"][s])
        if self._events is not None:
            state, grass = self._event_state()
            self._events.reset(state, self.agents, grass)
        return self._mask_dicts(out, obs), {}

    def step(self, action_dict):
        obs, rew, term, trunc, infos = super().step(action_dict)
        return self._mask_dicts(self._batch.outputs_numpy(), obs), rew, term, trunc, infos

    @property
    def agent_move_accumulator(self):
        acc = self._batch.read_env_acc(0)
        st = self._read()
        return {self._name(s, int(i)): float(v) for s in range(2) for i, v in zip(st["ids"][s], acc[s])}

    def _move_rate(self, speed):
        return 1.0 / self.max_cooldown + max(0.0, min(1.0, float(speed))) * (1.0 - 1.0 / self.max_cooldown)  # CAD:556-571

    def _cadence_keys(self, res, role, v):
        """the cadence keys that replace ECO's `fraction_fast` (CAD:524-542,1471-1485)"""
        res.pop(f"{role}_fraction_fast", None)
        if len(v):
            rates = np.array([self._move_rate(x) for x in v])
            cd = 1.0 / rates
            res[f"{role}_fraction_mobile"] = float(np.mean(rates >= 1.0 - 1e-9))
            res[f"{role}_fraction_fast_cadence"] = float(np.mean(cd <= max(1.0, self.max_cooldown / 2.0)))
            res[f"{role}_cooldown_mean"] = float(np.mean(cd))
        else:
            res[f"{role}_fraction_mobile"] = 0.0
            res[f"{role}_fraction_fast_cadence"] = 0.0
            res[f"{role}_cooldown_mean"] = float(self.max_cooldown)

    def episode_training_metrics(self):
        res = super().episode_training_metrics()
        for s, role in enumerate(("predator", "prey")):
            self._cadence_keys(res, role, self._episode_speeds[s])
        return res

    def live_speed_metrics(self):
        res = super().live_speed_metrics()
        st = self._read()
        for s, role in enumerate(("predator", "prey")):
            self._cadence_keys(res, role, st["speed"][s] if self.genome_enabled else [])
        return res


# ---------------------------------------------------------------------------------------------- STAG
class PredPreyGrassStag(_RowDictEnv):
    """stag_hunt_forward_view_nature_nurture `PredPreyGrass(config)`: mammoths and rabbits, join_hunt team capture,
    forward-shifted predator view, heritable cooperation trait."""

    _variant = VARIANT_STAG
    _stay = 4

    def __init__(self, config=None):
        super().__init__(config)
        c, g = self._cfg, config.get
        self.strict_rllib_output = bool(g("strict_rllib_output", False))  # STAG:126 (the device flag has the same default)
        self._n1 = (c.n_possible_t[0][0], c.n_possible_t[1][0])
        self.n_possible_type_1_predators, self.n_possible_type_2_predators = c.n_possible_t[0][0], c.n_possible_t[0][1]
        self.n_possible_type_1_prey, self.n_possible_type_2_prey = c.n_possible_t[1][0], c.n_possible_t[1][1]
        self.type_1_act_range, self.type_2_act_range = c.type_action_range[0], c.type_action_range[1]
        self.coop_trait_enabled = bool(c.coop_trait_enabled)
        self.possible_agents = ([f"type_1_predator_{i}" for i in range(c.n_possible_t[0][0])] +
                                [f"type_2_predator_{i}" for i in range(c.n_possible_t[0][1])] +
                                [f"type_1_prey_{i}" for i in range(c.n_possible_t[1][0])] +
                                [f"type_2_prey_{i}" for i in range(c.n_possible_t[1][1])])  # STAG:1768-1782
        C = self.num_obs_channels + (1 if self._vis_plane else 0)  # STAG:1788
        pred_space = Box(low=0, high=100.0, shape=(C, self.predator_obs_range, self.predator_obs_range), dtype=np.float32)
        prey_space = Box(low=0, high=100.0, shape=(C, self.prey_obs_range, self.prey_obs_range), dtype=np.float32)
        self.observation_spaces = {a: pred_space if "predator" in a else prey_space for a in self.possible_agents}
        sizes = {"type_1": max(1, self.type_1_act_range ** 2), "type_2": max(1, self.type_2_act_range ** 2)}
        self.action_spaces = {a: MultiDiscrete([sizes[a[:6]], 2]) if "predator" in a else Discrete(sizes[a[:6]])
                              for a in self.possible_agents}  # STAG:1800-1816
        self.observation_space = DictSpace(self.observation_spaces)
        self.action_space = DictSpace(self.action_spaces)
        self.predator_join_intent = {}

    def _vis(self, window, value):
        """include_visibility_channel (STAG:993-994): one more channel holding the reference's line-of-sight mask, which is
        all ones (see __init__); mask_observation_with_visibility multiplies by the same ones"""
        if not self._vis_plane:
            return window
        return np.concatenate([window, np.full((1,) + window.shape[1:], value, np.float32)])

    def _name(self, s, i):
        sp = "predator" if s == 0 else "prey"
        n1 = self._n1[s]
        return f"type_1_{sp}_{i}" if i < n1 else f"type_2_{sp}_{i - n1}"

    def _n_moves(self, agent):
        return max(1, (self.type_1_act_range if agent.startswith("type_1") else self.type_2_act_range) ** 2)

    def _action(self, s, value):
        """`_split_action` (STAG:771-799): predators pass [move, join_hunt] as array / tuple / dict; join defaults to 1"""
        if s == 1:
            return int(np.asarray(value).reshape(-1)[0]) if not isinstance(value, (int, np.integer)) else int(value)
        if isinstance(value, dict):
            move, join = int(value.get("move", 0)), int(value.get("join_hunt", 1))
        else:
            v = np.asarray(value).reshape(-1)
            move, join = int(v[0]), (int(v[1]) if v.size > 1 else 1)
        return move | ((1 if join else 0) << 8)

    def _unknown_actor(self, agent):
        # STAG:806-807 skips actions of agents that are no longer positioned (the ids that ended in the previous
        # step are still listed in `self.agents`, STAG:565-573, so callers do send them)
        if agent not in self.possible_agents:
            raise KeyError(agent)

    def _read(self):
        if self._state is None:
            self._state = self._batch.read_env_stag(0)
        return self._state

    def reset(self, *, seed=None, options=None):
        super().reset(seed=seed)
        if seed is None:
            seed = self.config.get("seed")
        if seed is None:
            seed = int(np.random.SeedSequence().generate_state(1, np.uint64)[0] >> 1)
        cells, facing, traits = reference_reset_tape_stag(seed, self.config)
        out = self._reset_device(seed, np.concatenate([cells, facing]), traits, options)
        self.predator_join_intent = {}
        obs = {}
        self._rows = {}
        for name, s, r, f in self._rows_of(out):  # founders: type_1/type_2 predators, type_1/type_2 prey (STAG:340-380)
            obs[name] = self._vis(out[f"obs{s}"][r], 1.0)
            self._rows[name] = (s, r)
        self.agents = list(obs)
        return obs, {}

    def step(self, action_dict):
        self.predator_join_intent = {}
        for a, v in action_dict.items():
            if "predator" in a and a in self._rows:
                self.predator_join_intent[a] = bool(self._action(0, v) >> 8)
        out = self._step_device({a: v for a, v in action_dict.items() if a in self._rows or a not in self.possible_agents})
        flags = int(out["env_flags"][0])
        rows = {name: (s, r, f) for name, s, r, f in self._rows_of(out)}
        ended = lambda f: bool(f & (ROW_TERMINATED | ROW_TRUNCATED))  # noqa: E731
        time_limit = bool(flags & ENV_TRUNCATED)
        extinct = bool(flags & ENV_TERMINATED)
        # self.agents: survivors in list order, then this step's newborns (predators, prey: STAG:490-496)
        live = [a for a in self.agents if a in rows and not (rows[a][2] & ROW_TERMINATED)]
        live += [a for a in rows if a not in self._rows and not (rows[a][2] & ROW_TERMINATED) and a not in live]
        gone = sorted(a for a in rows if a not in live)  # STAG:567-568
        obs, rew, term, trunc = {}, {}, {}, {}
        self.agents_just_ate = set()
        for a in live + gone:
            s, r, f = rows[a]
            obs[a] = self._vis(out[f"obs{s}"][r], 0.0 if f & ROW_TERMINATED else 1.0)  # ended agents: all-zero rows (STAG:596-612)
            rew[a] = float(out[f"reward{s}"][r])
            term[a] = bool(f & ROW_TERMINATED)
            trunc[a] = bool(f & ROW_TRUNCATED)
            if f & ROW_ATE:
                self.agents_just_ate.add(a)
        self._rows = {a: rows[a][:2] for a in live if not ended(rows[a][2])}
        self._state = None
        infos = self._infos(live + gone)
        term["__all__"] = extinct            # STAG:584-592
        trunc["__all__"] = time_limit        # STAG:659-716
        self.agents = live + gone if self.strict_rllib_output else live  # STAG:565-573
        if extinct or time_limit:
            self._done = True
        return obs, rew, term, trunc, infos

    def _infos(self, names):
        """STAG:498-546: the team-capture counters in every agent's info and in infos["__all__"]"""
        st = self._read()
        cap, capr = st["capture"], st["capture_real"]
        m_att, r_att = int(cap[4] + cap[5]), int(cap[6] + cap[7])
        common = {
            "team_capture_successes": int(cap[0]), "team_capture_failures": int(cap[1]),
            "team_capture_coop_successes": int(cap[2]), "team_capture_coop_failures": int(cap[3]),
            "team_capture_mammoth_successes": int(cap[4]), "team_capture_mammoth_failures": int(cap[5]),
            "team_capture_mammoth_success_rate": int(cap[4]) / m_att if m_att else 0.0,
            "team_capture_rabbit_successes": int(cap[6]), "team_capture_rabbit_failures": int(cap[7]),
            "team_capture_rabbit_success_rate": int(cap[6]) / r_att if r_att else 0.0,
        }
        trait = {self._name(0, int(i)): float(v) for i, v in zip(st["ids"][0], st["trait"])}
        infos = {}
        for a in names:
            info = dict(common)
            if "predator" in a:
                info["join_hunt"] = bool(self.predator_join_intent.get(a, True))
                info["coop_trait"] = trait.get(a, 0.0)
            infos[a] = info
        g = dict(common)
        g["team_capture_last_success_prob"] = float(capr[0])
        g["team_capture_last_effort_ratio"] = float(capr[1])
        g["team_capture_attempts"] = int(cap[8])
        g["team_capture_avg_success_prob"] = float(capr[2]) / int(cap[8]) if cap[8] > 0 else 0.0
        tv = np.asarray(st["trait"], np.float64)
        g["predator_mean_coop_trait"] = float(tv.mean()) if tv.size and self.coop_trait_enabled else 0.0
        g["predator_trait_variance"] = float(tv.var()) if tv.size and self.coop_trait_enabled else 0.0
        infos["__all__"] = g
        return infos

    def get_total_energy_by_type(self):
        """STAG:1964-1997: total energy of the live predators / prey (also per type) and of the grass"""
        totals = {"predator": 0.0, "prey": 0.0, "grass": sum(self.grass_energies.values()), "type_1_predator": 0.0,
                  "type_2_predator": 0.0, "type_1_prey": 0.0, "type_2_prey": 0.0}
        for agent, energy in self.agent_energies.items():
            role = "predator" if "predator" in agent else "prey"
            totals[role] += energy
            totals[("type_1_" if "type_1" in agent else "type_2_") + role] += energy
        return totals

    # STAG attributes
    @property
    def active_num_predators(self):
        return len(self._read()["ids"][0])

    @property
    def active_num_prey(self):
        return len(self._read()["ids"][1])

    @property
    def predator_facing(self):
        st = self._read()
        return {self._name(0, int(i)): FACING_OPTIONS[int(f)] for i, f in zip(st["ids"][0], st["facing"])}

    @property
    def predator_cooperation_trait(self):
        st = self._read()
        return {self._name(0, int(i)): float(v) for i, v in zip(st["ids"][0], st["trait"])}
