"""Row links on the GPU (`-m gpu`, include/ppg.h ppg_track_links): after every output prev_row equals, bit for bit, the numpy
reference of tests/test_links_cpu.py fed the oracle's outputs in lockstep; the other paths to an output (ordered and host
steps, the one-kernel step, queued ppg_rollout_random), switching on mid-run, snapshot / restore, non-interference with the
outputs and the launch count, the error paths; and the recurrent runner and state recording of connector.py."""
import numpy as np
import pytest

from predpreygrass_b200.config import BASE_CONFIG, ECO_CONFIG, STAG_CONFIG, TRAIT_CONFIGS, VARIANT_ECO, VARIANT_STAG, make_config
from tests.test_gae_cpu import life_sequences, snapshot
from tests.test_links_cpu import prev_rows

pytestmark = pytest.mark.gpu

ENV_TERM, ENV_TRUNC, ENV_RESET, ENV_IDLE = 0x01, 0x02, 0x04, 0x08


def _padded(a):
    A = np.zeros(max(1, len(a)), np.int32)
    A[: len(a)] = a
    return A


def _check(g, o0, o1, where):
    """the device's prev_row of output o1 (numpy columns) against the reference given the output o0 before it"""
    want = prev_rows(o0, o1)
    pr = g.prev_row()
    for s in range(2):
        got = pr[s][: o1["n"][s]].cpu().numpy()
        if not np.array_equal(got, want[s]):
            bad = np.nonzero(got != want[s])[0][:5]
            raise AssertionError(f"{where}: prev_row{s} differs at rows {bad.tolist()}: gpu={got[bad].tolist()} "
                                 f"reference={want[s][bad].tolist()}")
    assert int(g.links_error().item()) == 0, where
    return sum(int((w >= 0).sum()) for w in want)


def _lockstep(cfg, n_envs, steps, *, mask_at=None, action_seed=31):
    """GPU (links on before the reset) and oracle stepped with the same Philox actions; prev_row checked after every output.
    mask_at: before that step every third env's reset is scheduled on both sides, and prev_row must still describe the last
    output between the masked reset and the step."""
    import torch

    from oracle.oracle import Oracle
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    g, ora = BatchedPredPreyGrass(cfg, n_envs), Oracle(cfg, n_envs, threads=8)
    seen = {"flags": 0, "linked": 0}
    try:
        g.track_links(True)
        g.reset()
        prev = snapshot(ora.reset())
        pr = g.prev_row()
        assert all(bool((pr[s][: prev["n"][s]] == -1).all()) for s in range(2))  # a full reset: founders only
        for t in range(1, steps + 1):
            if t == mask_at:
                before = [p.clone() for p in g.prev_row()]
                mask = (np.arange(n_envs) % 3 == 0).astype(np.uint8)
                g.reset(mask=mask)
                ora.reset(mask=mask)
                assert all(before[s].equal(g.prev_row()[s]) for s in range(2))  # a masked reset only schedules
            a0, a1 = g.random_actions(action_seed)
            o0, o1 = ora.random_actions(action_seed)
            g.step(a0, a1)
            cur = snapshot(ora.step(_padded(o0), _padded(o1)))
            for s in range(2):
                assert np.array_equal(g.out.row_agent[s][: cur["n"][s]].cpu().numpy(), cur[f"row_agent{s}"]), (t, s)
            seen["linked"] += _check(g, prev, cur, f"output {t}")
            seen["flags"] |= int(np.bitwise_or.reduce(cur["env_flags"]))
            prev = cur
        torch.cuda.synchronize()
        return seen
    finally:
        g.close()
        ora.close()


# ------------------------------------------------------------------------------------------------ bit-exact against the reference
def test_links_base_4096_envs():
    seen = _lockstep(make_config(dict(BASE_CONFIG, max_steps=45), cap_live=(64, 192), seed=11), 4096, 60)
    assert seen["flags"] & ENV_TERM and seen["flags"] & ENV_TRUNC and seen["linked"] > 100000, seen


def test_links_add():
    assert _lockstep(make_config(dict(BASE_CONFIG, max_steps=30), reward_mode="additive", cap_live=(64, 192), seed=3), 512, 60)["flags"] & ENV_TRUNC


def test_links_eco_crowded_and_pool_exhausted():
    from tests.test_agent_state_cpu import _eco_carcasses
    from tests.test_returns_cpu import REUSE_CONFIG

    assert _lockstep(make_config(dict(_eco_carcasses(), max_steps=45), variant=VARIANT_ECO, cap_live=(96, 192), seed=17), 256, 90)["flags"] & ENV_TERM
    assert _lockstep(REUSE_CONFIG(), 128, 90)["flags"] & ENV_TRUNC


@pytest.mark.parametrize("trait", ["metabolic", "investment", "cooperation", "cadence"])
def test_links_trait_variants(trait):
    cfg = make_config(dict(TRAIT_CONFIGS[trait], max_steps=50), variant=VARIANT_ECO, cap_live=(64, 160), seed=7)
    assert _lockstep(cfg, 256, 80)["flags"] & (ENV_TERM | ENV_TRUNC)


def test_links_stag_bench_caps_walls_and_not_strict():
    from tests.test_gpu_parity_stag import CROWDED

    cfg = make_config(dict(STAG_CONFIG, max_steps=60, n_initial_active_type_1_predator=2), variant=VARIANT_STAG, cap_live=(160, 640), seed=6)
    assert _lockstep(cfg, 512, 80)["flags"] & ENV_TRUNC
    walls = [(3, y) for y in range(2, 8)] + [(6, 1), (6, 2), (7, 7), (8, 7), (1, 8), (9, 9)]
    cfg = dict(CROWDED, grid_size=10, manual_wall_positions=walls, respect_los_for_movement=True, type_2_action_range=5, max_steps=50)
    assert _lockstep(make_config(cfg, variant=VARIANT_STAG, cap_live=(96, 224), seed=31), 256, 70)["flags"] & (ENV_TERM | ENV_TRUNC)
    cfg = make_config(dict(STAG_CONFIG, max_steps=40, strict_rllib_output=False), variant=VARIANT_STAG, cap_live=(64, 192), seed=6)
    assert _lockstep(cfg, 256, 60)["flags"] & (ENV_TERM | ENV_TRUNC)


def test_links_masked_reset():
    assert _lockstep(make_config(dict(BASE_CONFIG, max_steps=40), cap_live=(64, 192), seed=5), 256, 30, mask_at=12)["flags"] & ENV_RESET
    cfg = make_config(dict(ECO_CONFIG, max_steps=40), variant=VARIANT_ECO, cap_live=(64, 128), seed=5)
    assert _lockstep(cfg, 128, 30, mask_at=9)["flags"] & ENV_RESET


def test_links_autoreset_off_idle_envs():
    cfg = make_config(dict(BASE_CONFIG, max_steps=20), cap_live=(64, 192), seed=3, autoreset=False)
    assert _lockstep(cfg, 128, 40)["flags"] & ENV_IDLE


def test_links_one_kernel_step(monkeypatch):
    """PPG_OBS_SPLIT=0 (read by ppg_create): the step kernel writes the rows and every ag_prow itself"""
    from predpreygrass_b200._lib import PpgError
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    monkeypatch.setenv("PPG_OBS_SPLIT", "0")
    cfg = make_config(dict(BASE_CONFIG, max_steps=30), cap_live=(64, 192), seed=4)
    probe = BatchedPredPreyGrass(cfg, 8)
    probe.reset()
    with pytest.raises(PpgError, match="one-kernel"):  # this handle really runs the one-kernel step
        probe.world_state()
    probe.close()
    seen = _lockstep(cfg, 256, 60)
    assert seen["flags"] & ENV_RESET and seen["linked"] > 0


# ------------------------------------------------------------------------------------------------ other paths to an output
def _gpu_out(g):
    return {k: v for k, v in g.outputs_numpy().items() if not k.startswith("obs")}


def test_links_step_ordered_and_step_host():
    """ppg_step_ordered with a shuffled order per env and ppg_step_host: the reference runs on the device's own consecutive
    outputs (the parity suites pin those to the oracle's)"""
    import torch

    from predpreygrass_b200.batched import BatchedPredPreyGrass

    cfg = make_config(dict(BASE_CONFIG, max_steps=25), cap_live=(64, 192), seed=2)
    g = BatchedPredPreyGrass(cfg, 256)
    rng = np.random.default_rng(1)
    g.track_links(True)
    g.reset()
    prev, linked = _gpu_out(g), 0
    for t in range(30):
        g.random_actions(7)
        orders = []
        for s in range(2):
            env = prev[f"row_env{s}"]
            o = np.zeros(max(1, len(env)), np.int32)
            for e in np.unique(env):
                r = np.nonzero(env == e)[0]
                o[r] = rng.permutation(len(r))
            orders.append(torch.from_numpy(o).to(g.device))
        g.step_ordered(g.actions[0], g.actions[1], orders[0], orders[1])
        cur = _gpu_out(g)
        linked += _check(g, prev, cur, f"ordered {t}")
        prev = cur
    host = g.make_host_buffers()
    for t in range(30):
        for s in range(2):
            host[f"actions{s}"].copy_(g.random_actions(5)[s].cpu())
        g.step_host(host)
        cur = _gpu_out(g)
        linked += _check(g, prev, cur, f"step_host {t}")
        prev = cur
    assert linked > 10000
    g.close()


@pytest.mark.parametrize("groups,chain", [(1, 0), (1, 1), (2, 0)])
def test_links_after_queued_rollout_random(groups, chain):
    """20 queued steps of ppg_rollout_random: the final output's prev_row against the oracle's outputs 19 and 20"""
    import torch

    from oracle.oracle import Oracle
    from predpreygrass_b200 import _lib
    from predpreygrass_b200.pipelined import PipelinedPredPreyGrass
    from tests.test_gpu_rollout import _factory

    B, K, seed = 512, 20, 4321
    factory = _factory("eco")
    before = _lib.load().ppg_set_pdl_chain(chain)
    try:
        pipe = PipelinedPredPreyGrass(factory, B, groups=groups)
        for e in pipe.envs:
            e.track_links(True)
        torch.cuda.synchronize()
        pipe.reset()
        pipe.rollout_random(K, seed)
        torch.cuda.synchronize()
        per = B // groups
        for gi, g in enumerate(pipe.envs):
            ora = Oracle(factory(gi * per), per, threads=8)
            try:
                ora.reset(None)
                outs = []
                for _ in range(K):
                    o0, o1 = ora.random_actions(seed)
                    outs.append(snapshot(ora.step(_padded(o0), _padded(o1))))
                assert _check(g, outs[-2], outs[-1], f"group {gi} chain {chain}") > 0
            finally:
                ora.close()
        pipe.close()
    finally:
        _lib.load().ppg_set_pdl_chain(before)


# ------------------------------------------------------------------------------------------------ switching, restore, isolation
def test_links_switched_on_mid_run_and_after_restore():
    from predpreygrass_b200._lib import PpgError
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    cfg = make_config(dict(ECO_CONFIG, max_steps=30), variant=VARIANT_ECO, cap_live=(64, 128), seed=3)
    g = BatchedPredPreyGrass(cfg, 128)
    with pytest.raises(PpgError, match="off"):
        g.prev_row()
    g.reset()
    for _ in range(7):
        g.step(*g.random_actions(2))
    g.track_links(True)
    with pytest.raises(PpgError, match="no output"):
        g.prev_row()
    prev = _gpu_out(g)
    g.step(*g.random_actions(2))
    cur = _gpu_out(g)
    assert _check(g, prev, cur, "first output after the switch-on") > 0  # the very next output is linked
    g.track_links(True)  # already on: nothing changes
    assert _check(g, prev, cur, "switched on twice") > 0
    # snapshot, some more steps, restore, step: the links point into the output the restore leaves in the buffers
    blob = g.snapshot()
    for _ in range(5):
        g.step(*g.random_actions(4))
    g.restore(blob)
    with pytest.raises(PpgError, match="ppg_restore"):
        g.prev_row()
    restored = _gpu_out(g)
    g.step(*g.random_actions(4))
    assert _check(g, restored, _gpu_out(g), "first output after restore") > 0
    # off: PpgError, on again: linked from the next output on
    g.track_links(False)
    with pytest.raises(PpgError, match="off"):
        g.prev_row()
    g.step(*g.random_actions(5))
    g.track_links(True)
    prev = _gpu_out(g)
    g.step(*g.random_actions(5))
    assert _check(g, prev, _gpu_out(g), "switched on again") > 0
    g.close()


def test_links_change_no_output_and_one_launch_per_output():
    from predpreygrass_b200.batched import BatchedPredPreyGrass
    from tests.parity import compare_outputs

    cfg = make_config(dict(STAG_CONFIG, max_steps=25), variant=VARIANT_STAG, cap_live=(64, 192), seed=8)
    a, b = BatchedPredPreyGrass(cfg, 256), BatchedPredPreyGrass(cfg, 256)
    n0 = a.launch_count()
    a.track_links(False)  # off: nothing launched or allocated
    assert a.launch_count() == n0
    a.track_links(True)
    assert a.launch_count() == n0 + 1  # the save-only launch
    base = a.launch_count() - b.launch_count()
    a.reset(); b.reset()
    for t in range(40):
        a.step(*a.random_actions(9))
        b.step(*b.random_actions(9))
        compare_outputs(a.outputs_numpy(), b.outputs_numpy(), f"step {t}")
    assert a.launch_count() - b.launch_count() - base == 41  # one per output: the reset and 40 steps
    a.track_links(False)
    n = a.launch_count() - b.launch_count()
    a.step(*a.random_actions(9)); b.step(*b.random_actions(9))
    assert a.launch_count() - b.launch_count() == n
    a.close(); b.close()


def test_links_error_paths():
    import ctypes as C

    import torch

    from predpreygrass_b200 import _lib
    from predpreygrass_b200.batched import BatchedPredPreyGrass
    from predpreygrass_b200.config import LINK_ERR_MISSING

    L = _lib.load()
    g = BatchedPredPreyGrass(make_config(BASE_CONFIG, cap_live=(64, 192), seed=1), 64)
    rows, err = (C.c_void_p * 2)(), C.c_void_p()
    assert L.ppg_get_links(g.h, C.byref(rows), C.byref(err)) == 4  # PPG_ERR_STATE: off
    assert L.ppg_get_links(g.h, None, C.byref(err)) == 1
    g.track_links(True)
    g.reset()
    g.step(*g.random_actions(1))
    assert int(g.links_error().item()) == 0
    # a corrupted row id (malformed state): no fault, the row stays unlinked and the sticky bit is set
    n_old = int(g.out.n_rows[0].item())
    assert n_old > 0
    g.out.row_agent[0][0] = 60000
    torch.cuda.synchronize()
    g.track_links(False)
    g.track_links(True)  # saves the tables from the lists: the corrupted row no longer matches its list entry
    g.step(*g.random_actions(1))
    torch.cuda.synchronize()
    assert int(g.links_error().item()) & LINK_ERR_MISSING
    pr = g.prev_row()[0][:n_old].cpu().numpy()
    assert (pr >= -1).all()
    g.links_error().zero_()
    g.step(*g.random_actions(1))
    assert int(g.links_error().item()) == 0
    g.close()


# ------------------------------------------------------------------------------------------------ recurrent runner
class _CounterPolicy:
    """state [id, counter]: state_out = [the row's id, counter + 1]; logits constant"""

    state_size = 2

    def __init__(self, env, s, n_logits):
        self.env, self.s, self.n_logits, self.seen = env, s, n_logits, []

    def __call__(self, obs, state_in):
        import torch

        k = obs.shape[0]
        ids = self.env.out.row_agent[self.s][:k].to(torch.float32)
        self.seen.append(state_in.clone())
        return torch.zeros((k, self.n_logits), device=obs.device), torch.stack([ids, state_in[:, 1] + 1], 1)


@pytest.mark.parametrize("variant", ["base", "eco", "stag"])
def test_recurrent_runner_carries_state_along_each_life(variant):
    """for every row of a valid env (returns tracking on): on linked rows state_in[:, 0] is the row's own id, and the counter
    is row_life - 1 on every row, over several hundred steps with auto-resets"""
    from predpreygrass_b200.batched import BatchedPredPreyGrass
    from predpreygrass_b200.connector import DeviceRollout
    from tests.test_gpu_rollout import _factory

    g = BatchedPredPreyGrass(_factory(variant)(0), 256)
    nl = [g.n_actions(0) + (2 if variant == "stag" else 0), g.n_actions(1)]
    pol = [_CounterPolicy(g, s, nl[s]) for s in range(2)]
    g.track_returns(True)
    runner = DeviceRollout(g, pol, seed=3, recurrent=True)
    g.reset()
    checked = linked = 0
    for t in range(300):
        runner.act()  # pol[s].seen[-1]: the state_in of the rows of the current output
        ret = g.returns()
        n = g.out.counts()
        pr = g.prev_row()
        for s in range(2):
            st = pol[s].seen[-1].cpu().numpy()
            valid = ret.env_valid.cpu().numpy()[g.out.row_env[s][: n[s]].cpu().numpy()] == 1
            life = ret.row_life[s][: n[s]].cpu().numpy()
            ids = g.out.row_agent[s][: n[s]].cpu().numpy()
            lk = pr[s][: n[s]].cpu().numpy() >= 0
            assert np.array_equal(st[valid, 1], life[valid] - 1), (variant, t, s)
            assert np.array_equal(st[valid & lk, 0], ids[valid & lk]), (variant, t, s)
            checked += int(valid.sum())
            linked += int((valid & lk).sum())
        g.step()
    assert checked > 10000 and linked > 5000
    assert int(g.links_error().item()) == 0
    g.close()


def test_gru_rollout_columns_sequences_and_carry():
    """a recurrent rollout recorded with keep_state: seq_id / seq_pos match the lives rebuilt on the host from the recorded
    ids and flags, state_in equals the runner's, and after carry() the next rollout's segments start from the carried state"""
    import torch

    from predpreygrass_b200.batched import BatchedPredPreyGrass
    from predpreygrass_b200.connector import DeviceRollout, GRUPolicy, RolloutBuffer

    cfg = make_config(dict(BASE_CONFIG, max_steps=20), cap_live=(64, 192), seed=5)
    g = BatchedPredPreyGrass(cfg, 64)
    n_in = [g.C * g.R[s] * g.R[s] for s in range(2)]
    pols = [GRUPolicy(n_in[s], 9, g.device, state_size=8, seed=s) for s in range(2)]
    vfs = [lambda obs, h: h.sum(1) for _ in range(2)]
    runner = DeviceRollout(g, pols, seed=1, recurrent=True)
    g.reset()
    T = 30
    buf = RolloutBuffer(g, T, keep_obs=False, keep_state=True)
    states = []
    orig_act = runner.act

    def act():
        res = orig_act()
        states.append(tuple(x.clone() for x in runner.state_in))
        return res

    runner.act = act
    for rollout in range(2):
        states.clear()
        runner.rollout(buf, vfs)
        buf.compute(0.99, 0.95)
        cols = buf.columns()
        outputs = []
        for t in range(T + 1):
            nr = buf.n_rows[t].tolist()
            o = {"n": (nr[0] + nr[2], nr[1] + nr[3]), "n_old": (nr[0], nr[1]), "env_flags": buf.env_flags[t].cpu().numpy()}
            for s in range(2):
                for c in ("row_env", "row_agent", "flags"):
                    o[f"{c}{s}"] = getattr(buf, c)[s][t, : o["n"][s]].cpu().numpy()
            outputs.append(o)
        for s, name in enumerate(("predator", "prey")):
            c = cols[name]
            cap = g.row_capacity[s]
            got = {}
            for sid, pos, st in zip(c["seq_id"].tolist(), c["seq_pos"].tolist(), c["state_in"].cpu()):
                got.setdefault(sid, []).append((pos, st))
            want = {}
            for seq in life_sequences(outputs, s):
                tr = [(t, r) for t, r in seq[:-1]]  # the transitions of the life (its last row has no successor)
                # a life the rollout cuts at a masked or automatic reset still splits where next_row is -1
                want[tr[0][0] * cap + tr[0][1]] = tr
            assert sorted(got) == sorted(want), (rollout, s)
            for sid, tr in want.items():
                assert [p for p, _ in got[sid]] == list(range(len(tr))), (rollout, s, sid)
                for (t, r), (_, st) in zip(tr, got[sid]):
                    assert torch.equal(st, states[t][s][r].cpu()), (rollout, s, t, r)
        if rollout == 1:  # the carried output's rows continue from the state the first rollout ended with
            assert all(torch.equal(states[0][s], carried[s]) for s in range(2))
        if rollout == 0:
            carried = tuple(x.clone() for x in runner.state_in)
            buf.carry()
            assert all(torch.equal(buf.state[0][s], carried[s]) for s in range(2))
    g.close()
