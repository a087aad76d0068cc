"""GAE advantages and value targets on the GPU (`-m gpu`, include/ppg.h ppg_gae): the device's adv, value_target and next_row
equal, bit for bit, the numpy reference of tests/test_gae_cpu.py fed the oracle's outputs of the same steps with the same
values.  Also the error paths, non-interference with the outputs and the launch count, and DeviceRollout.rollout end to end,
checked on a twin handle that replays the recorded actions."""
import numpy as np
import pytest

from predpreygrass_b200.config import (BASE_CONFIG, ECO_CONFIG, STAG_CONFIG, TRAIT_CONFIGS, VARIANT_ECO, VARIANT_STAG,
                                       make_config)
from tests.test_gae_cpu import (CONSERVATION_CASES, REUSE_CONFIG, _end_of_life, gae_reference, snapshot, synth_values)

pytestmark = pytest.mark.gpu

ROW_ENDED, ROW_FOUNDER, ROW_NEWBORN = 0x03, 0x08, 0x04


def _padded(a):
    A = np.zeros(max(1, len(a)), np.int32)
    A[: len(a)] = a
    return A


def _same_f32(got, want, where):
    got, want = np.asarray(got, np.float32), np.asarray(want, np.float32)
    gn, wn = np.isnan(got), np.isnan(want)
    if not np.array_equal(gn, wn) or not np.array_equal(got[~gn].view(np.uint32), want[~wn].view(np.uint32)):
        bad = np.argwhere((gn != wn) | ((got != want) & ~gn))[:5]
        raise AssertionError(f"{where}: differs at {bad.tolist()}: gpu={got[tuple(bad.T)]} reference={want[tuple(bad.T)]}")


def _lockstep_gae(cfg, n_envs, T, *, rollouts=1, preroll=0, mask_at=None, gamma=0.99, lam=0.95, action_seed=21):
    """GPU and oracle stepped with the same Philox actions; the GPU's outputs recorded into a RolloutBuffer with the synthetic
    values of the oracle's rows, the reference fed the oracle's outputs; rollouts > 1 are joined by carry()"""
    import torch

    from oracle.oracle import Oracle
    from predpreygrass_b200.batched import BatchedPredPreyGrass
    from predpreygrass_b200.connector import RolloutBuffer

    g, ora = BatchedPredPreyGrass(cfg, n_envs), Oracle(cfg, n_envs, threads=8)
    flags = 0
    try:
        g.reset()
        out = ora.reset()
        for _ in range(preroll):
            a0, a1 = g.random_actions(action_seed)
            o0, o1 = ora.random_actions(action_seed)
            g.step(a0, a1)
            out = ora.step(_padded(o0), _padded(o1))
            flags |= int(np.bitwise_or.reduce(out["env_flags"]))
        buf = RolloutBuffer(g, T, keep_obs=False)
        step = 0
        for k in range(rollouts):
            outs = [snapshot(out)]
            vals = [synth_values(out, step)]
            buf.record(tuple(torch.from_numpy(v).to(g.device) for v in vals[0]))
            for t in range(T):
                if mask_at is not None and step == mask_at:
                    mask = (np.arange(n_envs) % 3 == 0).astype(np.uint8)
                    g.reset(mask=mask)
                    ora.reset(mask=mask)
                a0, a1 = g.random_actions(action_seed)
                o0, o1 = ora.random_actions(action_seed)
                g.step(a0, a1)
                out = ora.step(_padded(o0), _padded(o1))
                step += 1
                flags |= int(np.bitwise_or.reduce(out["env_flags"]))
                outs.append(snapshot(out))
                vals.append(synth_values(out, step))
                buf.record(tuple(torch.from_numpy(v).to(g.device) for v in vals[-1]))
            buf.compute(gamma, lam)
            ref = gae_reference(outs, vals, gamma, lam)
            cols = buf.columns()  # raises on a flagged error; checks the recorded row counts
            for s in range(2):
                for t in range(T):
                    n = outs[t]["n"][s]
                    where = f"rollout {k} species {s} t {t}"
                    assert np.array_equal(buf.next_row[s][t, :n].cpu().numpy(), ref[s]["next_row"][t]), where
                    _same_f32(buf.advantages[s][t, :n].cpu().numpy(), ref[s]["adv"][t], where + " adv")
                    _same_f32(buf.value_targets[s][t, :n].cpu().numpy(), ref[s]["value_target"][t], where + " value_target")
                name = ("predator", "prey")[s]
                assert cols[name]["advantages"].shape[0] == sum(int((ref[s]["next_row"][t] >= 0).sum()) for t in range(T))
                assert not torch.isnan(cols[name]["advantages"]).any()
            if k + 1 < rollouts:
                buf.carry()
        return flags
    finally:
        g.close()
        ora.close()


# ------------------------------------------------------------------------------------------------ bit-exact against the reference
def test_gae_base_4096_envs():
    flags = _lockstep_gae(make_config(dict(BASE_CONFIG, max_steps=45), cap_live=(64, 192), seed=11), 4096, 64, preroll=36)
    assert flags & 1 and flags & 2  # episodes end by extinction and by time limit


def test_gae_add():
    _lockstep_gae(make_config(dict(BASE_CONFIG, max_steps=30), reward_mode="additive", cap_live=(64, 192), seed=3), 512, 48)


@pytest.mark.parametrize("case", ["crowded", "id_pool_exhausted"])
def test_gae_eco(case):
    cfg = CONSERVATION_CASES["eco_crowded"]() if case == "crowded" else REUSE_CONFIG()
    _lockstep_gae(cfg, 256, 64, gamma=0.95, lam=0.9)


def test_gae_stag_bench_caps():
    cfg = make_config(dict(STAG_CONFIG, max_steps=60, n_initial_active_type_1_predator=2), variant=VARIANT_STAG, cap_live=(160, 640), seed=6)
    assert _lockstep_gae(cfg, 512, 80) & 2


def test_gae_trait_variant():
    _lockstep_gae(make_config(dict(TRAIT_CONFIGS["metabolic"], max_steps=50), variant=VARIANT_ECO, cap_live=(64, 160), seed=7), 256, 60)


def test_gae_masked_reset():
    flags = _lockstep_gae(make_config(dict(BASE_CONFIG, max_steps=40), cap_live=(64, 192), seed=5), 256, 40, mask_at=13)
    assert flags & 4


def test_gae_autoreset_off():
    flags = _lockstep_gae(make_config(dict(BASE_CONFIG, max_steps=20), cap_live=(64, 192), seed=3, autoreset=False), 256, 40)
    assert flags & 8


def test_gae_two_rollouts_joined_by_carry():
    _lockstep_gae(make_config(dict(ECO_CONFIG, max_steps=40), variant=VARIANT_ECO, cap_live=(64, 128), seed=5), 256, 24, rollouts=2)
    _lockstep_gae(make_config(dict(BASE_CONFIG, max_steps=30), cap_live=(64, 192), seed=4), 512, 20, rollouts=3, gamma=1.0, lam=1.0)


# ------------------------------------------------------------------------------------------------ errors
def test_gae_error_paths():
    import ctypes as C

    import torch

    from predpreygrass_b200 import _lib
    from predpreygrass_b200.batched import BatchedPredPreyGrass
    from predpreygrass_b200.config import GAE_ERR_ID, GAE_ERR_LINK, PpgGaeArgs
    from predpreygrass_b200.connector import RolloutBuffer

    cfg = make_config(dict(BASE_CONFIG, max_steps=30), cap_live=(64, 192), seed=3)
    g = BatchedPredPreyGrass(cfg, 64)
    try:
        g.reset()
        buf = RolloutBuffer(g, 4)
        for t in range(5):
            n = g.out.counts()
            buf.record(tuple(torch.zeros(n[s], device=g.device) for s in range(2)))
            if t < 4:
                g.step(*g.random_actions(3))
        with pytest.raises(RuntimeError):
            buf.columns()  # before compute()
        with pytest.raises(RuntimeError):
            buf.record(buf.values)  # all outputs recorded
        # the C-ABI's argument checks
        L = _lib.load()
        stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

        def args(T=4, gamma=0.9, lam=0.9, null=None):
            a = PpgGaeArgs()
            a.T, a.gamma, a.lam = T, gamma, lam
            for f in ("row_agent", "flags", "reward", "old_off", "new_off", "new_cnt", "next_row"):
                for s in range(2):
                    getattr(a, f)[s] = getattr(buf, f)[s].data_ptr()
            for f, src in (("value", buf.values), ("adv", buf.advantages), ("value_target", buf.value_targets)):
                for s in range(2):
                    getattr(a, f)[s] = src[s].data_ptr()
            a.env_flags, a.error = buf.env_flags.data_ptr(), buf.error.data_ptr()
            if null:
                getattr(a, null)[1] = None
            return a

        assert L.ppg_gae(g.h, C.byref(args()), stream) == 0
        assert L.ppg_gae(g.h, None, stream) == 1
        for bad in (dict(T=0), dict(T=-3), dict(gamma=1.5), dict(lam=-0.1), dict(gamma=float("nan")), dict(null="value"),
                    dict(null="next_row")):
            assert L.ppg_gae(g.h, C.byref(args(**bad)), stream) == 1, bad
        a = args()
        a.error = None
        assert L.ppg_gae(g.h, C.byref(a), stream) == 1
        with pytest.raises(_lib.PpgError):
            g.gae(1.5, 0.9, buf.row_agent, buf.flags, buf.reward, buf.values, buf.old_off, buf.new_off, buf.new_cnt,
                  buf.env_flags, buf.advantages, buf.value_targets, buf.next_row, buf.error)
        with pytest.raises(ValueError):  # shapes and dtypes
            g.gae(0.9, 0.9, buf.row_agent, buf.flags, buf.reward, (buf.values[0].double(), buf.values[1]), buf.old_off,
                  buf.new_off, buf.new_cnt, buf.env_flags, buf.advantages, buf.value_targets, buf.next_row, buf.error)
        buf.compute(0.9, 0.9)
        buf.columns()
        assert int(buf.error) == 0
        # an id outside the pool, and an old row of output 2 without its predecessor in output 1: flagged, no fault
        keep = buf.row_agent[0].clone()
        buf.row_agent[0][1, 0] = int(cfg.n_possible[0]) + 5
        buf.compute(0.9, 0.9)
        with pytest.raises(_lib.PpgError):
            buf.columns()
        assert int(buf.error) & GAE_ERR_ID
        buf.row_agent[0].copy_(keep)
        buf.flags[0][1].fill_(0x01)  # every predator row of output 1 TERMINATED: the old rows of output 2 lose their predecessors
        buf.compute(0.9, 0.9)
        assert int(buf.error) & GAE_ERR_LINK
    finally:
        g.close()


# ------------------------------------------------------------------------------------------------ non-interference
def test_recording_leaves_outputs_and_launch_count_unchanged():
    import torch

    from predpreygrass_b200.batched import BatchedPredPreyGrass
    from predpreygrass_b200.connector import RolloutBuffer

    cfg = make_config(dict(BASE_CONFIG, max_steps=25), cap_live=(64, 192), seed=9)
    a, b = BatchedPredPreyGrass(cfg, 512), BatchedPredPreyGrass(cfg, 512)
    try:
        a.reset()
        b.reset()
        buf = RolloutBuffer(a, 10)
        computes = 0
        for t in range(31):
            n = a.out.counts()
            buf.record(tuple(torch.ones(n[s], device=a.device) for s in range(2)))
            if buf.t == buf.T + 1:
                buf.compute(0.99, 0.95)
                computes += 1
                buf.columns()
                buf.carry()
                buf.record(tuple(torch.ones(n[s], device=a.device) for s in range(2)))  # slot 0: the same output
            a.step(*a.random_actions(5))
            b.step(*b.random_actions(5))
            for f in ("obs", "row_env", "row_agent", "reward", "flags", "old_off", "new_off", "new_cnt"):
                for s in range(2):
                    assert torch.equal(getattr(a.out, f)[s], getattr(b.out, f)[s]), (t, f, s)
            for f in ("n_rows", "env_flags", "env_status", "env_step", "env_count"):
                assert torch.equal(getattr(a.out, f), getattr(b.out, f)), (t, f)
        assert computes == 3 and a.launch_count() == b.launch_count() + computes
    finally:
        a.close()
        b.close()


# ------------------------------------------------------------------------------------------------ DeviceRollout.rollout end to end
def _cfg(variant):
    if variant == "base":  # few founders: episodes end by extinction inside the rollout
        return make_config(dict(BASE_CONFIG, max_steps=60, n_initial_active_predator=2, n_initial_active_prey=3), cap_live=(32, 128), seed=3)
    if variant == "eco":  # crowded: episodes end by extinction; ECO flags the survivors TERMINATED
        from tests.test_gpu_parity_eco import CROWDED

        return make_config(dict(CROWDED, max_steps=60), variant=VARIANT_ECO, cap_live=(64, 64), seed=5)
    return make_config(dict(STAG_CONFIG, max_steps=50, n_initial_active_type_1_predator=2), variant=VARIANT_STAG, cap_live=(64, 192), seed=3)


@pytest.mark.parametrize("variant", ["base", "eco", "stag"])
def test_rollout_columns_replay_on_a_twin_handle(variant):
    """a twin handle of the same config replays the recorded (env, id, action) triples step by step; the rewards and
    end-of-life flags it reports for every transition equal those of columns(), and so do the observations"""
    import torch

    from predpreygrass_b200.batched import BatchedPredPreyGrass
    from predpreygrass_b200.connector import DeviceRollout, LinearPolicy, RolloutBuffer

    cfg, B, T = _cfg(variant), 96, 50
    a, b = BatchedPredPreyGrass(cfg, B), BatchedPredPreyGrass(cfg, B)
    try:
        a.reset()
        b.reset()
        n_logits = [a.n_actions(0) + (2 if variant == "stag" else 0), a.n_actions(1)]
        pols = [LinearPolicy(a.C * a.R[s] ** 2, n_logits[s], device=a.device, seed=11 + s) for s in range(2)]
        heads = [LinearPolicy(a.C * a.R[s] ** 2, 1, device=a.device, seed=31 + s) for s in range(2)]
        ro = DeviceRollout(a, pols, sample=True, seed=5)
        buf = ro.rollout(RolloutBuffer(a, T), heads)
        buf.compute(0.99, 0.95)
        cols = buf.columns()
        names = ("predator", "prey")
        want = {nm: {k: [] for k in ("obs", "rewards", "terminateds", "truncateds", "eps_id", "agent_index")} for nm in names}
        extinct_terminal = 0
        for t in range(T):
            before = b.out
            n = before.counts()
            obs = [before.obs[s][: n[s]].clone() for s in range(2)]
            env0 = [before.row_env[s][: n[s]].to(torch.int64) for s in range(2)]
            id0 = [before.row_agent[s][: n[s]].to(torch.int64) for s in range(2)]
            f0 = [before.flags[s][: n[s]].clone() for s in range(2)]
            for s in range(2):
                assert torch.equal(before.row_agent[s][: n[s]], buf.row_agent[s][t, : n[s]]), (variant, t, s)
                b.actions[s][: n[s]] = buf.actions[s][t, : n[s]]
            out = b.step()
            for s, nm in enumerate(names):
                k1 = out.n_rows[s].item()
                f1 = out.flags[s][:k1]
                ok = (f1 & (ROW_FOUNDER | ROW_NEWBORN)) == 0
                key1 = out.row_env[s][:k1].to(torch.int64) * 65536 + out.row_agent[s][:k1].to(torch.int64)
                rows1 = torch.nonzero(ok).squeeze(1)
                key1s, order = torch.sort(key1[rows1])
                rows1 = rows1[order]
                live = ((f0[s] & ROW_ENDED) == 0) & ((out.env_flags[env0[s]] & 0x0C) == 0)
                r0 = torch.nonzero(live).squeeze(1)
                key0 = env0[s][r0] * 65536 + id0[s][r0]
                pos = torch.searchsorted(key1s, key0).clamp(max=max(len(key1s) - 1, 0))
                hit = key1s[pos] == key0 if len(key1s) else torch.zeros_like(key0, dtype=torch.bool)
                assert int(hit.sum()) == len(key1s), (variant, t, nm)  # every old, non-FOUNDER row has its predecessor
                r0, r1 = r0[hit], rows1[pos[hit]]
                term, trunc = _end_of_life(f1[r1].cpu().numpy(), out.env_flags[env0[s][r0]].cpu().numpy())
                w = want[nm]
                w["obs"].append(obs[s][r0])
                w["rewards"].append(out.reward[s][r1])
                w["terminateds"].append(torch.from_numpy(term).to(a.device))
                w["truncateds"].append(torch.from_numpy(trunc).to(a.device))
                w["eps_id"].append(env0[s][r0])
                w["agent_index"].append(id0[s][r0])
                ext = ((out.env_flags[env0[s][r0]] & 0x01) != 0).cpu().numpy()
                extinct_terminal += int(ext.sum())
                if variant != "stag":
                    assert term[ext].all(), (variant, t, nm)  # survivors of an extinction are terminal transitions
        for nm in names:
            for k, v in want[nm].items():
                assert torch.equal(torch.cat(v), cols[nm][k]), (variant, nm, k)
            c = cols[nm]
            m = c["obs"].shape[0]
            assert all(c[k].shape[0] == m for k in ("actions", "action_logp", "vf_preds", "advantages", "value_targets"))
            assert not torch.isnan(c["advantages"]).any() and bool((c["action_logp"] <= 0).all())
            assert torch.equal(c["value_targets"], c["advantages"] + c["vf_preds"])
        if variant != "stag":
            assert extinct_terminal > 0, variant  # the rollout saw extinctions
        assert torch.equal(a.out.n_rows, b.out.n_rows) and torch.equal(a.out.env_step, b.out.env_step)
    finally:
        a.close()
        b.close()
