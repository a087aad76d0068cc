"""Zero-copy consumer path (SURVEY §8f3): the compact CUDA row batches go straight into a torch policy and the actions
come straight back — no per-agent dicts, no host copy of observations.

The reference trains with RLlib PPO, one policy per species (`policy_mapping_fn`: agent id prefix -> "predator" /
"prey" policy, eco_evolutionary/tune_ppo.py:42-51), each a `DefaultPPOTorchRLModule` whose encoder is the conv stack
of `eco_evolutionary/utils/networks.py:6-76`.  RLlib's `MultiAgentEnvRunner` would call `env.step(action_dict)` once per
env and build those per-policy batches from dicts; here a step already IS the per-policy batch:

    out.obs[s][:n]   float32 [n, C, R_s, R_s]   every agent of species s of every env, one row each
    env.actions[s]   int32   [cap]              the policy writes row i's action at index i

`DeviceRollout` is the env-runner loop over that layout; `collect()` returns per-policy column dicts with RLlib's
column names (`obs`, `actions`, `rewards`, `terminateds`, `truncateds`, `eps_id`, `agent_index`, `action_logp`) as
CUDA tensors, ready for a learner.  ray is not importable in this image, so the hand-over to an actual
`MultiRLModule` is shown in INTEGRATION.md, not executed here.  torch is the consumer here, not the product: the
environment step stays in the CUDA kernels.

`RolloutBuffer` records T+1 outputs of a handle (`DeviceRollout.rollout()` fills it) and computes PPO's GAE advantages and
value targets over them with one `ppg_gae` kernel launch (include/ppg.h); `columns()` hands out the transitions under
RLlib's names, `advantages` and `value_targets` included.

Recurrent policies: `DeviceRollout(..., recurrent=True)` switches the env's row links on (include/ppg.h ppg_track_links) and
carries each agent's hidden state from its row in one output to its row in the next with one gather per species;
`RolloutBuffer(..., keep_state=True)` records the state each action was computed from and marks each agent's life segment
(`seq_id`, `seq_pos`) so a learner can cut BPTT sequences.
"""
import torch

from .config import VARIANT_STAG

ROW_TERMINATED, ROW_TRUNCATED, ROW_NEWBORN, ROW_FOUNDER = 0x01, 0x02, 0x04, 0x08
ENV_TERMINATED, ENV_TRUNCATED = 0x01, 0x02
STAG_JOIN_SHIFT = 8


class LinearPolicy(torch.nn.Module):
    """the smallest stochastic policy: logits = W · flatten(obs) + b (a stand-in that exercises the plumbing)"""

    def __init__(self, n_in, n_out, device, seed=0):
        super().__init__()
        g = torch.Generator(device="cpu").manual_seed(seed)
        self.lin = torch.nn.Linear(n_in, n_out)
        with torch.no_grad():
            self.lin.weight.copy_(torch.randn(n_out, n_in, generator=g) * 0.05)
            self.lin.bias.zero_()
        self.to(device)

    def forward(self, obs):
        return self.lin(obs.flatten(1))


class GRUPolicy(torch.nn.Module):
    """the smallest recurrent policy: a linear encoder, a GRU cell, a logits head (a stand-in that exercises the plumbing of
    DeviceRollout(recurrent=True)).  forward(obs [n, C, R, R], state_in [n, state_size]) -> (logits, state_out)"""

    def __init__(self, n_in, n_out, device, state_size=16, seed=0):
        super().__init__()
        torch.manual_seed(seed)
        self.state_size = state_size
        self.enc = torch.nn.Linear(n_in, state_size)
        self.cell = torch.nn.GRUCell(state_size, state_size)
        self.head = torch.nn.Linear(state_size, n_out)
        self.to(device)

    def forward(self, obs, state_in):
        h = self.cell(torch.relu(self.enc(obs.flatten(1))), state_in)
        return self.head(h), h


class ConvPolicy(torch.nn.Module):
    """the reference's module shape (networks.py:28-50): L = (R - 1) // 2 conv layers 3x3 stride 1 with 16, 32, 64, 64...
    filters, then fully connected [256, 256] (or [384, 256] for > 20 actions), ReLU, a logits head"""

    def __init__(self, channels, window, n_out, device):
        super().__init__()
        L = (window - 1) // 2
        widths = ([16, 32, 64] + [64] * max(0, L - 3))[:L]
        layers, c = [], channels
        for w in widths:
            layers += [torch.nn.Conv2d(c, w, 3, stride=1, padding=1), torch.nn.ReLU()]  # RLlib pads "same"
            c = w
        self.conv = torch.nn.Sequential(*layers)
        hid = [384, 256] if n_out > 20 else [256, 256]
        self.fc = torch.nn.Sequential(torch.nn.Linear(c * window * window, hid[0]), torch.nn.ReLU(), torch.nn.Linear(hid[0], hid[1]),
                                      torch.nn.ReLU(), torch.nn.Linear(hid[1], n_out))
        self.to(device)

    def forward(self, obs):
        return self.fc(self.conv(obs).flatten(1))


class DeviceRollout:
    """env-runner loop on the device: policy(obs rows) -> actions in place -> ppg_step.

    policies: (predator_module, prey_module); a module maps float32 [n, C, R, R] to logits [n, n_logits].  For the STAG
    predator (`MultiDiscrete([n_moves, 2])`, STAG:1813-1816) the logits are n_moves + 2 wide: move logits, then join_hunt logits.

    recurrent=True: each module has a `state_size` attribute H and is called as module(obs, state_in) -> (logits, state_out)
    with state_in float32 [n, H].  The runner switches the env's row links on and keeps each species' state_out of the last
    forward; the next state_in of a row is the state_out of the row its agent had in the previous output (env.prev_row()),
    zeros for founders and newborns.  `state_in` holds the (pred, prey) states of the last act().
    """

    def __init__(self, env, policies, stream=None, sample=True, seed=0, recurrent=False):
        self.env, self.policies, self.stream, self.sample = env, policies, stream, sample
        self.gen = torch.Generator(device=env.device).manual_seed(seed)
        self.variant = env.cfg.variant
        self.last = None
        self.recurrent = recurrent
        if recurrent:
            env.track_links(True)
            self.state_out = [None, None]  # state_out of the last forward per species, rows of the output it ran on
            self.state_in = (None, None)

    def _ctx(self):
        return torch.cuda.stream(self.stream) if self.stream is not None else torch.cuda.stream(torch.cuda.current_stream(self.env.device))

    def _pick(self, logits):
        if not self.sample:
            return logits.argmax(-1), None
        logp = torch.log_softmax(logits, -1)
        a = torch.multinomial(logp.exp(), 1, generator=self.gen).squeeze(1)
        return a, logp.gather(1, a.unsqueeze(1)).squeeze(1)

    @torch.no_grad()
    def act(self):
        """policy forward on the rows of the last output; actions written into env.actions in place.
        -> per species (n, actions int64 [n], logp or None)"""
        env, out = self.env, self.env.out
        n = out.counts()  # 16 bytes device -> host: the row counts of the last output
        if self.recurrent:
            self.state_in = self._next_state_in(n)
        res = []
        for s in range(2):
            k = n[s]
            if k == 0:
                if self.recurrent:
                    self.state_out[s] = self.state_in[s]
                res.append((0, None, None))
                continue
            if self.recurrent:
                logits, self.state_out[s] = self.policies[s](out.obs[s][:k], self.state_in[s])
            else:
                logits = self.policies[s](out.obs[s][:k])
            if self.variant == VARIANT_STAG and s == 0:
                nm = env.n_actions(0)
                mv, lp1 = self._pick(logits[:, :nm])
                jn, lp2 = self._pick(logits[:, nm:nm + 2])
                a = mv | (jn << STAG_JOIN_SHIFT)
                lp = None if lp1 is None else lp1 + lp2
            else:
                a, lp = self._pick(logits)
            env.actions[s][:k] = a.to(torch.int32)
            res.append((k, a, lp))
        return res

    def _next_state_in(self, n):
        """(pred, prey) float32 [n_s, H]: the state_out of each row's agent in the previous output, zeros where unlinked"""
        res, prev = [], None
        for s in range(2):
            H, so = self.policies[s].state_size, self.state_out[s]
            if so is None or so.shape[0] == 0 or n[s] == 0:  # nothing to carry: the first output, or no rows before
                res.append(torch.zeros((n[s], H), dtype=torch.float32, device=self.env.device))
                continue
            if prev is None:
                prev = self.env.prev_row()
            pr = prev[s][: n[s]].to(torch.int64)
            res.append(torch.where((pr >= 0)[:, None], so[pr.clamp(min=0)], 0.0))
        return tuple(res)

    @torch.no_grad()
    def step(self):
        with self._ctx():
            self.last = self.act()
            return self.env.step()

    @torch.no_grad()
    def rollout(self, buffer, value_fns):
        """fills `buffer` (a RolloutBuffer of this env, empty or just carried): T times act -> record -> step, then records
        output T.  value_fns: (predator, prey); each maps the observation rows float32 [n, C, R, R] to values [n]; a recurrent
        runner calls them as value_fn(obs, state_in) and hands state_in to the buffer (recorded with keep_state)."""
        if buffer.env is not self.env:
            raise ValueError("rollout: the buffer belongs to another env")
        with self._ctx():
            for _ in range(buffer.T):
                acted = self.act()
                buffer.record(self._values(acted, value_fns), actions=tuple(a for _, a, _ in acted),
                              logp=None if not self.sample else tuple(lp for _, _, lp in acted),
                              **({"state_in": self.state_in} if self.recurrent else {}))
                self.env.step()
                self.last = acted
            n = self.env.out.counts()
            if self.recurrent:
                self.state_in = self._next_state_in(n)
            buffer.record(self._values(tuple((n[s], None, None) for s in range(2)), value_fns),
                          **({"state_in": self.state_in} if self.recurrent else {}))
        return buffer

    def _values(self, acted, value_fns):
        out = self.env.out
        if self.recurrent:
            return tuple(value_fns[s](out.obs[s][:k], self.state_in[s]).reshape(-1) if k else torch.zeros(0, device=self.env.device)
                         for s, (k, _, _) in enumerate(acted))
        return tuple(value_fns[s](out.obs[s][:k]).reshape(-1) if k else torch.zeros(0, device=self.env.device)
                     for s, (k, _, _) in enumerate(acted))

    @torch.no_grad()
    def collect(self, n_steps, check=False):
        """n_steps of experience -> {"predator": columns, "prey": columns}.  A transition pairs the observation and action of
        an agent in output t with the reward / termination flags output t+1 reports for the same (env, agent id).  The rows of
        t+1 are grouped by env with last step's newborns merged in, so the pairing is a key match on the device (sort +
        gather), not a positional one.  Rows produced by reset() (ROW_FOUNDER) or born in t+1 (ROW_NEWBORN) have no
        predecessor; rows already terminated / truncated in t have no successor."""
        names = ("predator", "prey")
        cols = {nm: {k: [] for k in ("obs", "actions", "action_logp", "rewards", "terminateds", "truncateds", "eps_id", "agent_index")} for nm in names}
        npos = (int(self.env.cfg.n_possible[0]), int(self.env.cfg.n_possible[1]))
        with self._ctx():
            for _ in range(n_steps):
                prev = self.env.out
                acted = self.act()
                keep = []
                for s in range(2):
                    k, a, lp = acted[s]
                    if k == 0:
                        keep.append(None)
                        continue
                    live = (prev.flags[s][:k] & (ROW_TERMINATED | ROW_TRUNCATED)) == 0
                    key = prev.row_env[s][:k].to(torch.int64) * npos[s] + prev.row_agent[s][:k].to(torch.int64)
                    key, order = torch.sort(key[live])
                    keep.append((prev.obs[s][:k][live][order], a[live][order], None if lp is None else lp[live][order], key))
                out = self.env.step()
                n_old = out.n_rows[:2].tolist()
                for s, nm in enumerate(names):
                    if keep[s] is None:
                        continue
                    obs, a, lp, key = keep[s]
                    k2 = n_old[s]
                    f = out.flags[s][:k2]
                    succ = (f & ROW_FOUNDER) == 0
                    key2 = out.row_env[s][:k2].to(torch.int64) * npos[s] + out.row_agent[s][:k2].to(torch.int64)
                    key2, order2 = torch.sort(key2[succ])
                    if check:
                        assert key2.shape == key.shape and bool((key2 == key).all()), "row pairing broken"
                    c = cols[nm]
                    c["obs"].append(obs)
                    c["actions"].append(a)
                    if lp is not None:
                        c["action_logp"].append(lp)
                    c["rewards"].append(out.reward[s][:k2][succ][order2])
                    f2 = f[succ][order2]
                    c["terminateds"].append((f2 & ROW_TERMINATED) != 0)
                    c["truncateds"].append((f2 & ROW_TRUNCATED) != 0)
                    c["eps_id"].append(key // npos[s])
                    c["agent_index"].append(key % npos[s])
        return {nm: {k: (torch.cat(v) if v else None) for k, v in c.items()} for nm, c in cols.items()}


class RolloutBuffer:
    """T+1 consecutive outputs 0..T of one handle and the value estimates of their rows, on the device (include/ppg.h ppg_gae).

    Slot t of every slab holds output t: per species row_agent, row_env, flags, reward and `values` [T+1, cap] (rows [0, n_t)
    valid), old_off [T+1, B+1], new_off, new_cnt and env_flags [T+1, B]; actions and logp of the rows of output t [T, cap];
    the observation rows [n_t, C, R, R] of each output (keep_obs=False skips them).  `values` is public: a learner may
    overwrite it, e.g. with the value predictions of updated weights, and call compute() again.  Per step, record() only copies
    into these slabs, except that with keep_obs it clones each output's observation rows (one allocation per species).
    keep_state=True: record() also takes state_in = (pred, prey) [n_s, H], the recurrent state each row's action was computed
    from, and clones it the same way; columns() then adds state_in, seq_id and seq_pos."""

    def __init__(self, env, n_steps, keep_obs=True, keep_state=False):
        T = int(n_steps)
        if T < 1:
            raise ValueError("RolloutBuffer: n_steps must be >= 1")
        self.env, self.T, self.keep_obs, self.keep_state = env, T, keep_obs, keep_state
        d, B, cap = env.device, env.n_envs, env.row_capacity

        def slab(rows, n, dtype, fill=0):
            return tuple(torch.full((rows, n[s] if isinstance(n, tuple) else n), fill, dtype=dtype, device=d) for s in range(2))

        self.row_agent = slab(T + 1, cap, torch.int32)
        self.row_env = slab(T + 1, cap, torch.int32)
        self.flags = slab(T + 1, cap, torch.uint8)
        self.reward = slab(T + 1, cap, torch.float32)
        self.values = slab(T + 1, cap, torch.float32)
        self.old_off = slab(T + 1, B + 1, torch.int32)
        self.new_off = slab(T + 1, B, torch.int32)
        self.new_cnt = slab(T + 1, B, torch.int32)
        self.env_flags = torch.zeros((T + 1, B), dtype=torch.uint8, device=d)
        self.n_rows = torch.zeros((T + 1, 4), dtype=torch.int32, device=d)
        self.actions = slab(T, cap, torch.int32)
        self.logp = slab(T, cap, torch.float32)
        self.advantages = slab(T, cap, torch.float32)
        self.value_targets = slab(T, cap, torch.float32)
        self.next_row = slab(T, cap, torch.int32, -1)
        self.error = torch.zeros(1, dtype=torch.int32, device=d)
        self.obs = [[None, None] for _ in range(T + 1)]
        self.state = [[None, None] for _ in range(T + 1)]
        self.n = [(0, 0)] * (T + 1)  # rows of each output, from the length of its values
        self.t = 0                   # outputs recorded
        self.has_logp = False
        self._carried = False
        self._computed = False

    def record(self, values, actions=None, logp=None, state_in=None):
        """Records the env's current output into slot t: values = (v_pred, v_prey), float32 [n_s] for every row of the output
        (terminated and truncated rows included); actions / logp: (pred, prey) [n_s] of the rows of this output, for slots
        0..T-1; state_in (with keep_state; a carried slot keeps its state without it): (pred, prey) float32 [n_s, H].
        Tensor.copy_ on the current stream, no host synchronisation."""
        t, T, out = self.t, self.T, self.env.out
        if t > T:
            raise RuntimeError(f"RolloutBuffer.record: all {T + 1} outputs are recorded (compute, columns, then carry)")
        if self.keep_state and state_in is None and not self._carried:
            raise ValueError("RolloutBuffer.record: keep_state needs state_in")
        n = tuple(int(values[s].shape[0]) for s in range(2))
        for s in range(2):
            if n[s] > self.env.row_capacity[s]:
                raise ValueError(f"RolloutBuffer.record: {n[s]} values for species {s}, capacity {self.env.row_capacity[s]}")
            k = n[s]
            if not self._carried:
                self.row_agent[s][t, :k].copy_(out.row_agent[s][:k])
                self.row_env[s][t, :k].copy_(out.row_env[s][:k])
                self.flags[s][t, :k].copy_(out.flags[s][:k])
                self.reward[s][t, :k].copy_(out.reward[s][:k])
                self.old_off[s][t].copy_(out.old_off[s])
                self.new_off[s][t].copy_(out.new_off[s])
                self.new_cnt[s][t].copy_(out.new_cnt[s])
                self.obs[t][s] = out.obs[s][:k].clone() if self.keep_obs else None
            if self.keep_state and state_in is not None:
                self.state[t][s] = state_in[s][:k].clone()
            self.values[s][t, :k].copy_(values[s])
            if t < T and actions is not None and actions[s] is not None:
                self.actions[s][t, :k].copy_(actions[s])
            if t < T and logp is not None and logp[s] is not None:
                self.logp[s][t, :k].copy_(logp[s])
                self.has_logp = True
        if not self._carried:
            self.env_flags[t].copy_(out.env_flags)
            self.n_rows[t].copy_(out.n_rows)
        elif n != self.n[0]:
            raise ValueError(f"RolloutBuffer.record: the carried output has {self.n[0]} rows, got values for {n}")
        self.n[t] = n
        self.t, self._carried, self._computed = t + 1, False, False

    def compute(self, gamma, lam):
        """advantages and value_targets of every row from `values` (one ppg_gae launch, no synchronisation)"""
        if self.t != self.T + 1:
            raise RuntimeError(f"RolloutBuffer.compute: {self.t} of {self.T + 1} outputs recorded")
        self.env.gae(gamma, lam, self.row_agent, self.flags, self.reward, self.values, self.old_off, self.new_off, self.new_cnt,
                     self.env_flags, self.advantages, self.value_targets, self.next_row, self.error)
        self._computed = True

    @torch.no_grad()
    def columns(self):
        """{"predator": columns, "prey": columns}: one entry per transition (row (t, r) with next_row >= 0), ordered by t, then
        row, under RLlib's names: obs, actions, action_logp (None unless recorded), rewards, terminateds, truncateds (of the
        successor row, by the rule of include/ppg.h), vf_preds, advantages, value_targets, eps_id (env index) and agent_index
        (agent id).  With keep_state also state_in (the recorded state of the row), seq_id (int64: one id per agent life
        segment inside the rollout, the flat index t0 * cap + r0 of the segment's first row) and seq_pos (int32: the
        transition's position in its segment), derived from the links compute() produced; a learner cuts BPTT chunks of
        length L where seq_pos % L == 0 and starts each from state_in there.  Synchronises once; raises PpgError if the
        kernel flagged malformed slabs."""
        from ._lib import PpgError

        if not self._computed:
            raise RuntimeError("RolloutBuffer.columns: call compute() first")
        T, B, d = self.T, self.env.n_envs, self.env.device
        cap = self.env.row_capacity
        nr_dev = self.n_rows[:T].to(torch.int64)
        masks, counts = [], []
        for s in range(2):
            n_t = nr_dev[:, s] + nr_dev[:, s + 2]  # rows of each output: the slots beyond hold an earlier rollout's values
            m = (self.next_row[s] >= 0) & (torch.arange(cap[s], device=d)[None, :] < n_t[:, None])
            masks.append(m)
            counts.append(m.sum(1))
        host = torch.cat([self.error.to(torch.int64), counts[0], counts[1], self.n_rows.to(torch.int64).flatten()]).tolist()
        if host[0]:
            raise PpgError(f"ppg_gae flagged the recorded slabs: error bits {host[0]:#x} (include/ppg.h PPG_GAE_ERR_*)")
        nr = host[1 + 2 * T:]
        for t in range(T + 1):
            want = (nr[4 * t] + nr[4 * t + 2], nr[4 * t + 1] + nr[4 * t + 3])
            if want != self.n[t]:
                raise ValueError(f"RolloutBuffer: output {t} has {want} rows but values for {self.n[t]} were recorded")
        res = {}
        for s, name in enumerate(("predator", "prey")):
            per_t = host[1 + s * T: 1 + (s + 1) * T]
            total = sum(per_t)
            m = masks[s].flatten()
            pos = torch.cumsum(m, 0) - 1  # stable compaction without a synchronisation: slot `total` takes the rest
            idx = torch.empty(total + 1, dtype=torch.int64, device=d)
            idx.scatter_(0, torch.where(m, pos, total), torch.arange(m.numel(), device=d))
            i = idx[:total]
            t_i, r_i = i // cap[s], i % cap[s]
            j = (t_i + 1) * cap[s] + self.next_row[s].flatten()[i].to(torch.int64)
            env_i = self.row_env[s].flatten()[i].to(torch.int64)
            f1 = self.flags[s].flatten()[j]
            ef1 = self.env_flags.flatten()[(t_i + 1) * B + env_i]
            term = ((f1 & ROW_TERMINATED) != 0) | (((ef1 & ENV_TERMINATED) != 0) & ((f1 & ROW_TRUNCATED) == 0))
            trunc = ~term & (((f1 & ROW_TRUNCATED) != 0) | ((ef1 & ENV_TRUNCATED) != 0))
            obs = None
            if self.keep_obs:
                parts, k = [], 0
                for t in range(T):
                    if per_t[t]:
                        parts.append(self.obs[t][s][r_i[k:k + per_t[t]]])
                    k += per_t[t]
                obs = torch.cat(parts) if parts else self.obs[0][s][:0]
            extra = {}
            if self.keep_state:
                seg_id, seg_pos = self._segments(s)
                parts, k = [], 0
                for t in range(T):
                    if per_t[t]:
                        parts.append(self.state[t][s][r_i[k:k + per_t[t]]])
                    k += per_t[t]
                extra = {"state_in": torch.cat(parts) if parts else self.state[0][s][:0],
                         "seq_id": seg_id.flatten()[i], "seq_pos": seg_pos.flatten()[i]}
            res[name] = {
                "obs": obs,
                "actions": self.actions[s].flatten()[i].to(torch.int64),
                "action_logp": self.logp[s].flatten()[i] if self.has_logp else None,
                "rewards": self.reward[s].flatten()[j],
                "terminateds": term,
                "truncateds": trunc,
                "vf_preds": self.values[s].flatten()[i],
                "advantages": self.advantages[s].flatten()[i],
                "value_targets": self.value_targets[s].flatten()[i],
                "eps_id": env_i,
                "agent_index": self.row_agent[s].flatten()[i].to(torch.int64),
                **extra,
            }
        return res

    def _segments(self, s):
        """[T, cap] segment id and position of every row of outputs 0..T-1, forward along next_row: a row another row links
        to continues that row's segment, every other row starts one"""
        T, cap, d = self.T, self.env.row_capacity[s], self.env.device
        ar = torch.arange(cap, device=d)
        seg_id = torch.empty((T, cap), dtype=torch.int64, device=d)
        seg_pos = torch.zeros((T, cap), dtype=torch.int32, device=d)
        seg_id[0] = ar
        n_t = self.n_rows[:, s] + self.n_rows[:, s + 2]
        for t in range(T - 1):
            nr = self.next_row[s][t].to(torch.int64)
            dst = torch.where((nr >= 0) & (ar < n_t[t]), nr, cap)  # unlinked rows scatter into a spill slot
            sid = torch.cat([(t + 1) * cap + ar, ar[:1]])
            spos = torch.zeros(cap + 1, dtype=torch.int32, device=d)
            sid.scatter_(0, dst, seg_id[t])
            spos.scatter_(0, dst, seg_pos[t] + 1)
            seg_id[t + 1], seg_pos[t + 1] = sid[:cap], spos[:cap]
        return seg_id, seg_pos

    def carry(self):
        """makes output T slot 0 of the next rollout (its columns, values and observation rows); the next record() adds the
        actions of that output (and may replace its values) without copying the output again"""
        if self.t != self.T + 1:
            raise RuntimeError(f"RolloutBuffer.carry: {self.t} of {self.T + 1} outputs recorded")
        T = self.T
        for s in range(2):
            for sl in (self.row_agent, self.row_env, self.flags, self.reward, self.values, self.old_off, self.new_off, self.new_cnt):
                sl[s][0].copy_(sl[s][T])
            self.obs[0][s] = self.obs[T][s]
            self.state[0][s] = self.state[T][s]
        self.env_flags[0].copy_(self.env_flags[T])
        self.n_rows[0].copy_(self.n_rows[T])
        self.n[0] = self.n[T]
        self.obs[1:] = [[None, None] for _ in range(T)]
        self.state[1:] = [[None, None] for _ in range(T)]
        self.t, self._carried, self._computed, self.has_logp = 0, True, False, False
