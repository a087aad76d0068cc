"""BatchedPredPreyGrass — thousands of PredPreyGrass instances stepped in lockstep on one GPU.

Thin host layer over the C-ABI (include/ppg.h): it owns a handle, wraps the handle's device
buffers as torch tensors WITHOUT copying, and passes torch tensors' device pointers back in.  All
compute is in the CUDA kernels (csrc/); torch is only the allocator / stream / tensor view here.

Row model: see include/ppg.h.  `step(actions_pred, actions_prey)` takes one int32 action per row
of the previous output and returns a `StepOutput` of views.
"""
import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from .config import N_EP_STATS, N_STATS, STAT_NAMES, VARIANT_ECO, PpgBuffers, PpgConfig, PpgReturns, PpgTape


class _DevPtr:
    """zero-copy bridge: a raw device pointer exposed through __cuda_array_interface__"""

    def __init__(self, ptr, shape, typestr):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 3}


_TYPESTR = {torch.float32: "<f4", torch.float64: "<f8", torch.int32: "<i4", torch.uint8: "|u1", torch.int64: "<i8"}


def _view(ptr, shape, dtype, device):
    if int(np.prod(shape)) == 0:
        return torch.empty(shape, dtype=dtype, device=device)
    return torch.as_tensor(_DevPtr(ptr, shape, _TYPESTR[dtype]), device=device)


@dataclass
class StepOutput:
    """Views into the handle's output buffers; valid until the next reset()/step()."""

    obs: tuple          # (pred [cap0, C, R0, R0], prey [cap1, C, R1, R1]) fp32 — first n rows valid
    row_env: tuple      # int32 [cap]
    row_agent: tuple    # int32 [cap]
    reward: tuple       # fp32 [cap]
    flags: tuple        # uint8 [cap]  ROW_* bits
    old_off: tuple      # int32 [B+1]
    new_off: tuple      # int32 [B]  first newborn row of the env (defined where new_cnt > 0)
    new_cnt: tuple      # int32 [B]  newborn rows of the env
    n_rows: torch.Tensor   # int32 [4] on device: n_old_pred, n_old_prey, n_new_pred, n_new_prey
    env_flags: torch.Tensor
    env_status: torch.Tensor
    env_step: torch.Tensor
    env_count: torch.Tensor

    def counts(self):
        """(n_pred_rows, n_prey_rows) — synchronises (device -> host read of 16 bytes)."""
        n = self.n_rows.tolist()
        return n[0] + n[2], n[1] + n[3]


@dataclass
class Returns:
    """Views of the episode-returns state (include/ppg.h ppg_track_returns); the row columns belong to the last output."""

    row_return: tuple   # (pred, prey) f64 [cap]: return so far of the row's agent in this life
    row_life: tuple     # (pred, prey) int32 [cap]: rows so far of the row's agent in this life
    env_return: torch.Tensor  # f64 [B, 2]: running episode return per species (NaN: env not valid)
    env_valid: torch.Tensor   # uint8 [B]: 1 once the env has been reset since tracking was switched on / a restore
    env_acc: torch.Tensor     # f64 [B, N_EP_STATS]: each env's share of episode_stats_device()


def episode_metrics_from_stats(v):
    """The PPG_N_EP_STATS vector (summed over envs and ranks) -> RLlib's episode metric names, plus per-species lifetimes.
    Means are nan when their count is 0; with no episode, episode_return_max is -inf and episode_return_min +inf."""
    v = np.asarray(v, np.float64)
    if v.shape != (N_EP_STATS,):
        raise ValueError(f"expected the {N_EP_STATS}-slot episode statistics vector, got shape {v.shape}")

    def mean(total, count):
        return float(total / count) if count > 0 else float("nan")

    n = v[0]
    sp = ("predator", "prey")
    life = [v[8 + 4 * s: 12 + 4 * s] for s in range(2)]  # lives, deaths, return sum, rows sum
    return {
        "num_episodes": int(n),
        "episode_return_mean": mean(v[2], n),
        "episode_return_min": float(-v[7]),
        "episode_return_max": float(v[6]),
        "episode_len_mean": mean(v[1], n),
        "module_episode_returns_mean": {"predator": mean(v[4], n), "prey": mean(v[5], n)},
        "agent_lifetime_return_mean": {sp[s]: mean(life[s][2], life[s][0]) for s in range(2)},
        "agent_lifetime_rows_mean": {sp[s]: mean(life[s][3], life[s][0]) for s in range(2)},
        "agent_deaths": {sp[s]: int(life[s][1]) for s in range(2)},
        "agent_lives_ended": {sp[s]: int(life[s][0]) for s in range(2)},
    }


class BatchedPredPreyGrass:
    def __init__(self, cfg: PpgConfig, n_envs: int, device=0):
        if not torch.cuda.is_available():
            raise _lib.PpgError("BatchedPredPreyGrass needs a CUDA device (no CPU fallback)")
        self.L = _lib.load()
        self.cfg, self.n_envs = cfg, int(n_envs)
        self.device = torch.device("cuda", device if isinstance(device, int) else device.index or 0)
        h = C.c_void_p()
        rc = self.L.ppg_create(C.byref(cfg), self.n_envs, self.device.index, C.byref(h))
        _lib.check(rc)
        self.h = h
        b = PpgBuffers()
        _lib.check(self.L.ppg_get_buffers(self.h, C.byref(b)), self.h)
        # row channels: the grid channels, plus ECO's own-speed plane (ECO:707-711)
        self.C = (cfg.num_obs_channels + (1 if cfg.variant == VARIANT_ECO and cfg.include_speed_in_obs else 0)
                  + (1 if cfg.variant == 2 and cfg.include_visibility_channel else 0))  # STAG:1788
        self.R = (cfg.obs_range[0], cfg.obs_range[1])
        self.row_capacity = (int(b.row_capacity[0]), int(b.row_capacity[1]))
        d, B = self.device, self.n_envs
        cap = self.row_capacity
        self.out = StepOutput(
            obs=tuple(_view(b.obs[s], (cap[s], self.C, self.R[s], self.R[s]), torch.float32, d) for s in range(2)),
            row_env=tuple(_view(b.row_env[s], (cap[s],), torch.int32, d) for s in range(2)),
            row_agent=tuple(_view(b.row_agent[s], (cap[s],), torch.int32, d) for s in range(2)),
            reward=tuple(_view(b.reward[s], (cap[s],), torch.float32, d) for s in range(2)),
            flags=tuple(_view(b.flags[s], (cap[s],), torch.uint8, d) for s in range(2)),
            old_off=tuple(_view(b.old_off[s], (B + 1,), torch.int32, d) for s in range(2)),
            new_off=tuple(_view(b.new_off[s], (B,), torch.int32, d) for s in range(2)),
            new_cnt=tuple(_view(b.new_cnt[s], (B,), torch.int32, d) for s in range(2)),
            n_rows=_view(b.n_rows, (4,), torch.int32, d),
            env_flags=_view(b.env_flags, (B,), torch.uint8, d),
            env_status=_view(b.env_status, (B,), torch.uint8, d),
            env_step=_view(b.env_step, (B,), torch.int32, d),
            env_count=_view(b.env_count, (B, 2), torch.int32, d),
        )
        # action buffers a caller may use (any int32 CUDA tensor of >= n rows works)
        self.actions = tuple(torch.zeros(cap[s], dtype=torch.int32, device=d) for s in range(2))

    # ------------------------------------------------------------------ lifecycle
    def close(self):
        if getattr(self, "h", None):
            torch.cuda.synchronize(self.device)
            self.L.ppg_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    # ------------------------------------------------------------------ API
    def load_tape(self, cells_per_env, reals_per_env=None):
        """Replay tape (include/ppg.h ppg_tape): per env the recorded cells and, for ECO, the recorded real draws."""

        def flatten(seqs, dtype):
            off = np.zeros(self.n_envs + 1, np.int64)
            for i, c in enumerate(seqs):
                off[i + 1] = off[i] + len(c)
            flat = np.concatenate([np.asarray(c, dtype) for c in seqs]) if off[-1] else np.zeros(1, dtype)
            return np.ascontiguousarray(flat, dtype), off

        flat, off = flatten(cells_per_env, np.int32)
        t = PpgTape()
        t.cells = flat.ctypes.data_as(C.POINTER(C.c_int32))
        t.cell_off = off.ctypes.data_as(C.POINTER(C.c_int64))
        if reals_per_env is not None:
            rflat, roff = flatten(reals_per_env, np.float64)
            t.reals = rflat.ctypes.data_as(C.POINTER(C.c_double))
            t.real_off = roff.ctypes.data_as(C.POINTER(C.c_int64))
        _lib.check(self.L.ppg_load_tape(self.h, C.byref(t)), self.h)

    def reset(self, seeds=None, mask=None):
        s = None if seeds is None else np.ascontiguousarray(seeds, np.uint64)
        m = None if mask is None else np.ascontiguousarray(mask, np.uint8)
        rc = self.L.ppg_reset(self.h, None if s is None else s.ctypes.data, None if m is None else m.ctypes.data, self._stream())
        _lib.check(rc, self.h)
        if s is not None or m is not None:
            torch.cuda.current_stream(self.device).synchronize()  # host staging arrays must outlive the copy
        # a masked reset only SCHEDULES the reset: the masked envs are reset by the next step() (include/ppg.h), whose output
        # carries their founders' rows — there is no new output to hand out here
        return None if m is not None else self.out

    def step(self, actions_pred=None, actions_prey=None):
        a0 = self.actions[0] if actions_pred is None else actions_pred
        a1 = self.actions[1] if actions_prey is None else actions_prey
        assert a0.dtype == torch.int32 and a1.dtype == torch.int32 and a0.is_cuda and a1.is_cuda
        _lib.check(self.L.ppg_step(self.h, a0.data_ptr(), a1.data_ptr(), self._stream()), self.h)
        return self.out

    def step_ordered(self, actions_pred, actions_prey, order_pred, order_prey):
        """step() with an explicit action-dict iteration order: order_*[row] = position of the row's agent
        among its env's acting agents of that species (int32 CUDA tensors, a permutation per env)."""
        for t in (actions_pred, actions_prey, order_pred, order_prey):
            assert t.dtype == torch.int32 and t.is_cuda
        rc = self.L.ppg_step_ordered(self.h, actions_pred.data_ptr(), actions_prey.data_ptr(), order_pred.data_ptr(),
                                     order_prey.data_ptr(), self._stream())
        _lib.check(rc, self.h)
        return self.out

    def n_actions(self, s=0):
        """size of the movement action space of species s: 9 (BASE:96-106), action_range**2 (ECO:225-232), the type ranges (STAG:178-193)"""
        from .config import VARIANT_BASE

        if self.cfg.variant == VARIANT_BASE:
            return 9
        if self.cfg.variant == VARIANT_ECO:
            return int(self.cfg.action_range) ** 2
        return max(int(self.cfg.type_action_range[0]), int(self.cfg.type_action_range[1])) ** 2

    def random_actions(self, seed, out_pred=None, out_prey=None):
        a0 = self.actions[0] if out_pred is None else out_pred
        a1 = self.actions[1] if out_prey is None else out_prey
        _lib.check(self.L.ppg_random_actions(self.h, int(seed), a0.data_ptr(), a1.data_ptr(), self._stream()), self.h)
        return a0, a1

    def make_host_buffers(self, pinned=True):
        """Host-side row batch for step_host(): dict of pinned tensors + the ppg_buffers struct."""
        B, cap = self.n_envs, self.row_capacity
        mk = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=pinned)  # noqa: E731
        t = {}
        for s in range(2):
            t[f"obs{s}"] = mk((cap[s], self.C, self.R[s], self.R[s]), torch.float32)
            t[f"row_env{s}"] = mk((cap[s],), torch.int32)
            t[f"row_agent{s}"] = mk((cap[s],), torch.int32)
            t[f"reward{s}"] = mk((cap[s],), torch.float32)
            t[f"flags{s}"] = mk((cap[s],), torch.uint8)
            t[f"old_off{s}"] = mk((B + 1,), torch.int32)
            t[f"new_off{s}"] = mk((B,), torch.int32)
            t[f"new_cnt{s}"] = mk((B,), torch.int32)
            t[f"actions{s}"] = torch.zeros((cap[s],), dtype=torch.int32, pin_memory=pinned)
        t["env_flags"] = mk((B,), torch.uint8)
        t["env_status"] = mk((B,), torch.uint8)
        t["env_step"] = mk((B,), torch.int32)
        t["env_count"] = mk((B, 2), torch.int32)
        t["n_rows"] = torch.zeros(4, dtype=torch.int32)
        b = PpgBuffers()
        for s in range(2):
            b.obs[s] = t[f"obs{s}"].data_ptr(); b.row_env[s] = t[f"row_env{s}"].data_ptr()
            b.row_agent[s] = t[f"row_agent{s}"].data_ptr(); b.reward[s] = t[f"reward{s}"].data_ptr()
            b.flags[s] = t[f"flags{s}"].data_ptr(); b.old_off[s] = t[f"old_off{s}"].data_ptr()
            b.new_off[s] = t[f"new_off{s}"].data_ptr(); b.new_cnt[s] = t[f"new_cnt{s}"].data_ptr(); b.row_capacity[s] = cap[s]
        b.env_flags = t["env_flags"].data_ptr(); b.env_status = t["env_status"].data_ptr()
        b.env_step = t["env_step"].data_ptr(); b.env_count = t["env_count"].data_ptr()
        b.n_rows = t["n_rows"].data_ptr()
        b.n_envs = B
        t["_struct"] = b
        return t

    def step_host(self, host):
        """ppg_step_host: actions from host memory, row batch back into host memory (synchronises)."""
        rc = self.L.ppg_step_host(self.h, host["actions0"].data_ptr(), host["actions1"].data_ptr(), C.byref(host["_struct"]),
                                  host["n_rows"].data_ptr(), self._stream())
        _lib.check(rc, self.h)
        n = host["n_rows"].tolist()
        return n[0] + n[2], n[1] + n[3]

    def stats(self):
        out = np.zeros(N_STATS, np.int64)
        _lib.check(self.L.ppg_stats(self.h, out.ctypes.data, self._stream()), self.h)
        return dict(zip(STAT_NAMES, out.tolist()))

    def stats_device(self):
        p = C.c_void_p()
        _lib.check(self.L.ppg_stats_device(self.h, C.byref(p), self._stream()), self.h)
        return _view(p.value, (N_STATS,), torch.int64, self.device)

    def stats_clear(self):
        _lib.check(self.L.ppg_stats_clear(self.h, self._stream()), self.h)

    # ------------------------------------------------------------------ episode returns (include/ppg.h ppg_track_returns)
    def track_returns(self, on=True):
        """Switch episode-return tracking on or off.  Switching on marks every env invalid until its next reset, so call
        it before reset() to see every episode."""
        _lib.check(self.L.ppg_track_returns(self.h, 1 if on else 0, self._stream()), self.h)

    def returns(self):
        """Zero-copy views of the tracking state (a `Returns`); PpgError while tracking is off."""
        r = PpgReturns()
        _lib.check(self.L.ppg_get_returns(self.h, C.byref(r)), self.h)
        d, B, cap = self.device, self.n_envs, self.row_capacity
        return Returns(row_return=tuple(_view(r.row_return[s], (cap[s],), torch.float64, d) for s in range(2)),
                       row_life=tuple(_view(r.row_life[s], (cap[s],), torch.int32, d) for s in range(2)),
                       env_return=_view(r.env_return, (B, 2), torch.float64, d),
                       env_valid=_view(r.env_valid, (B,), torch.uint8, d),
                       env_acc=_view(r.env_acc, (B, N_EP_STATS), torch.float64, d))

    def episode_stats_device(self):
        """The N_EP_STATS float64 vector reduced over the valid envs, on the current stream without synchronising: a view of
        a buffer of the handle, valid until the next call."""
        p = C.c_void_p()
        _lib.check(self.L.ppg_episode_stats_device(self.h, C.byref(p), self._stream()), self.h)
        return _view(p.value, (N_EP_STATS,), torch.float64, self.device)

    def episode_stats_clear(self):
        _lib.check(self.L.ppg_episode_stats_clear(self.h, self._stream()), self.h)

    def episode_metrics(self, group=None):
        """RLlib's episode metrics over this handle's envs (and over the ranks of `group` when torch.distributed is
        initialised): episode_stats_device() all-reduced and converted by episode_metrics_from_stats.  Synchronises."""
        from .sharding import allreduce_episode_stats

        return episode_metrics_from_stats(allreduce_episode_stats(self.episode_stats_device().clone(), group).cpu().numpy())

    def launch_count(self):
        return int(self.L.ppg_launch_count(self.h))

    def profile_env_cycles(self):
        """-> (cycles, info, start_ns, sm), each [n_envs], of the last step-kernel launch (include/ppg.h)"""
        out = [np.zeros(self.n_envs, np.uint32) for _ in range(4)]
        _lib.check(self.L.ppg_profile_env_cycles(self.h, *[a.ctypes.data for a in out], self._stream()), self.h)
        return tuple(out)

    def profile_begin(self):
        """start timing the kernels of every step with CUDA events on the step's stream (include/ppg.h)"""
        _lib.check(self.L.ppg_profile_begin(self.h), self.h)

    def profile_end(self):
        """-> (ms in the step kernel, ms in the observation kernel, steps timed), summed since profile_begin"""
        a, b, n = C.c_double(), C.c_double(), C.c_int32()
        _lib.check(self.L.ppg_profile_end(self.h, C.byref(a), C.byref(b), C.byref(n)), self.h)
        return a.value, b.value, n.value

    def world_state(self, env_begin=0, n=None, out=None):
        """`grid_world_state` of envs [env_begin, env_begin + n) after the last output (include/ppg.h ppg_world_state):
        float32 CUDA tensor [n, num_obs_channels, G, G], written on the current stream without synchronising.  Without
        `out` it is a view of a buffer this object owns and reuses: valid until the next world_state() call."""
        n = self.n_envs - int(env_begin) if n is None else int(n)
        G, C = self.cfg.grid_size, self.cfg.num_obs_channels
        shape = (n, C, G, G)
        if out is None:
            if getattr(self, "_world", None) is None:
                self._world = torch.empty((self.n_envs, C, G, G), dtype=torch.float32, device=self.device)
            out = self._world[: max(n, 0)]
        elif out.dtype != torch.float32 or out.device != self.device or not out.is_contiguous() or tuple(out.shape) != shape:
            raise ValueError(f"world_state: out must be a contiguous float32 tensor of shape {shape} on {self.device}, got "
                             f"{out.dtype} {tuple(out.shape)} on {out.device} (contiguous={out.is_contiguous()})")
        _lib.check(self.L.ppg_world_state(self.h, int(env_begin), n, out.data_ptr(), self._stream()), self.h)
        return out

    def snapshot(self):
        n = self.L.ppg_snapshot_size(self.h)
        blob = np.empty(n, np.uint8)
        _lib.check(self.L.ppg_snapshot(self.h, blob.ctypes.data, n, self._stream()), self.h)
        return blob

    def restore(self, blob):
        blob = np.ascontiguousarray(blob, np.uint8)
        _lib.check(self.L.ppg_restore(self.h, blob.ctypes.data, blob.size, self._stream()), self.h)

    def read_env(self, env):
        cap = (self.cfg.cap_live[0], self.cfg.cap_live[1])
        n = np.zeros(2, np.int32)
        ids = [np.zeros(cap[s], np.int32) for s in range(2)]
        xy = [np.zeros((cap[s], 2), np.int32) for s in range(2)]
        en = [np.zeros(cap[s], np.float64) for s in range(2)]
        ng = max(1, self.cfg.n_grass)
        gxy, ge = np.zeros((ng, 2), np.int32), np.zeros(ng, np.float64)
        rc = self.L.ppg_read_env(self.h, env, n.ctypes.data, ids[0].ctypes.data, xy[0].ctypes.data, en[0].ctypes.data,
                                 ids[1].ctypes.data, xy[1].ctypes.data, en[1].ctypes.data, gxy.ctypes.data, ge.ctypes.data)
        _lib.check(rc, self.h)
        return {"ids": (ids[0][: n[0]], ids[1][: n[1]]), "xy": (xy[0][: n[0]], xy[1][: n[1]]),
                "energy": (en[0][: n[0]], en[1][: n[1]]), "grass_xy": gxy[: self.cfg.n_grass], "grass_energy": ge[: self.cfg.n_grass]}

    def read_env_eco(self, env):
        """read_env plus the ECO attributes agent_ages, genome speeds, dead_prey, active_num_* (ECO:153,177,193,212)."""
        st = self.read_env(env)
        n = (len(st["ids"][0]), len(st["ids"][1]))
        age = [np.zeros(max(1, n[s]), np.int32) for s in range(2)]
        sp = [np.zeros(max(1, n[s]), np.float64) for s in range(2)]
        dead = np.zeros(max(1, n[1]), np.uint8)
        act = np.zeros(2, np.int32)
        rc = self.L.ppg_read_env_eco(self.h, env, age[0].ctypes.data, sp[0].ctypes.data, age[1].ctypes.data, sp[1].ctypes.data,
                                     dead.ctypes.data, act.ctypes.data)
        _lib.check(rc, self.h)
        st.update(age=(age[0][: n[0]], age[1][: n[1]]), speed=(sp[0][: n[0]], sp[1][: n[1]]), dead_prey=dead[: n[1]], active_num=act)
        return st

    def read_env_acc(self, env):
        """CAD `agent_move_accumulator` of the live agents of one env, in the order of read_env (include/ppg.h ppg_read_env_acc)"""
        n = self.read_env(env)["ids"]
        acc = [np.zeros(max(1, len(n[s])), np.float64) for s in range(2)]
        _lib.check(self.L.ppg_read_env_acc(self.h, env, acc[0].ctypes.data, acc[1].ctypes.data), self.h)
        return tuple(a[: len(n[s])] for s, a in enumerate(acc))

    def read_episode_eco(self, env):
        """per-episode totals of one ECO env (include/ppg.h ppg_read_episode_eco; needs make_config(track_episode_sums=True)):
        -> {"distance": (pred, prey), "move_energy": (pred, prey), "spawned": (pred, prey)}"""
        sums, sp = np.zeros(4, np.float64), np.zeros(2, np.int32)
        _lib.check(self.L.ppg_read_episode_eco(self.h, env, sums.ctypes.data, sp.ctypes.data), self.h)
        return {"distance": (float(sums[0]), float(sums[1])), "move_energy": (float(sums[2]), float(sums[3])), "spawned": (int(sp[0]), int(sp[1]))}

    def read_episode_events_eco(self, env):
        """event counters of the running episode of one trait-variant env (include/ppg.h ppg_read_episode_events_eco):
        -> {"blocked_capacity": (pred, prey), "blocked_density": n, "satiation_blocked": n, "donated": (pred, prey)}"""
        ev = np.zeros(6, np.float64)
        _lib.check(self.L.ppg_read_episode_events_eco(self.h, env, ev.ctypes.data), self.h)
        return {"blocked_capacity": (int(ev[0]), int(ev[1])), "blocked_density": int(ev[2]), "satiation_blocked": int(ev[3]),
                "donated": (float(ev[4]), float(ev[5]))}

    def read_env_stag(self, env):
        """read_env (lists in `self.agents` insertion order) plus the STAG attributes agent_ages, predator_facing (index into
        `_predator_facing_options`, STAG:197-206), predator_cooperation_trait and the team-capture counters (STAG:237-254)."""
        st = self.read_env(env)
        n = (len(st["ids"][0]), len(st["ids"][1]))
        age = [np.zeros(max(1, n[s]), np.int32) for s in range(2)]
        face = np.zeros(max(1, n[0]), np.int32)
        trait = np.zeros(max(1, n[0]), np.float64)
        cap = np.zeros(12, np.int64)
        capr = np.zeros(3, np.float64)
        rc = self.L.ppg_read_env_stag(self.h, env, age[0].ctypes.data, face.ctypes.data, trait.ctypes.data, age[1].ctypes.data,
                                      cap.ctypes.data, capr.ctypes.data)
        _lib.check(rc, self.h)
        st.update(age=(age[0][: n[0]], age[1][: n[1]]), facing=face[: n[0]], trait=trait[: n[0]], capture=cap, capture_real=capr)
        return st

    def outputs_numpy(self):
        """Host copy (numpy) of the valid part of the last output."""
        o = self.out
        n = o.n_rows.tolist()
        res = {"n_old": (n[0], n[1]), "n_new": (n[2], n[3]), "n": (n[0] + n[2], n[1] + n[3])}
        for s in range(2):
            k = res["n"][s]
            res[f"obs{s}"] = o.obs[s][:k].cpu().numpy()
            res[f"row_env{s}"] = o.row_env[s][:k].cpu().numpy()
            res[f"row_agent{s}"] = o.row_agent[s][:k].cpu().numpy()
            res[f"reward{s}"] = o.reward[s][:k].cpu().numpy()
            res[f"flags{s}"] = o.flags[s][:k].cpu().numpy()
            res[f"old_off{s}"] = o.old_off[s].cpu().numpy()
            res[f"new_off{s}"] = o.new_off[s].cpu().numpy()
            res[f"new_cnt{s}"] = o.new_cnt[s].cpu().numpy()
        res["env_flags"] = o.env_flags.cpu().numpy()
        res["env_status"] = o.env_status.cpu().numpy()
        res["env_step"] = o.env_step.cpu().numpy()
        res["env_count"] = o.env_count.cpu().numpy()
        return res
