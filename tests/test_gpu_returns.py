"""Episode returns and agent lifetimes on the GPU (`-m gpu`, include/ppg.h ppg_track_returns): after every output the
device's row columns, per-env returns, validity bytes and accumulators equal, bit for bit, the numpy tracker of
tests/test_returns_cpu.py fed the oracle's outputs of the same steps.  Also the aggregate vector, the lifecycle (masked
reset, switch-on mid-run, snapshot and restore, the error state, ppg_step_host), queued rollouts with the launch chain off
and on, non-interference with the outputs and the launch count, and sharding over env_index_base."""
import numpy as np
import pytest

from predpreygrass_b200.config import (BASE_CONFIG, ECO_CONFIG, STAG_CONFIG, VARIANT_BASE, VARIANT_ECO, VARIANT_STAG,
                                       make_config)
from tests.test_returns_cpu import CONSERVATION_CASES, REUSE_CONFIG, Tracker

pytestmark = pytest.mark.gpu


def _same_f64(got, want, where):
    """bit-identical, NaN wherever the other side is NaN (the device's NaN bits may differ from numpy's)"""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    gn, wn = np.isnan(got), np.isnan(want)
    if not np.array_equal(gn, wn) or not np.array_equal(got[~gn].view(np.uint64), want[~wn].view(np.uint64)):
        bad = np.argwhere((gn != wn) | ((got != want) & ~gn))[:5]
        raise AssertionError(f"{where}: differs at {bad.tolist()}: gpu={got[tuple(bad.T)]} tracker={want[tuple(bad.T)]}")


def _compare(g, tr, n, where):
    r = g.returns()
    for s in range(2):
        _same_f64(r.row_return[s][: n[s]].cpu().numpy(), tr.row_return[s], f"{where} row_return{s}")
        assert np.array_equal(r.row_life[s][: n[s]].cpu().numpy(), tr.row_life[s]), f"{where} row_life{s}"
    _same_f64(r.env_return.cpu().numpy(), tr.env_return, f"{where} env_return")
    assert np.array_equal(r.env_valid.cpu().numpy(), tr.env_valid), f"{where} env_valid"
    _same_f64(r.env_acc.cpu().numpy(), tr.env_acc, f"{where} env_acc")


def _padded(a):
    A = np.zeros(max(1, len(a)), np.int32)
    A[: len(a)] = a
    return A


def _lockstep(cfg, n_envs, steps, *, on_at=-1, mask_at=None, action_seed=21, every=1):
    """GPU and oracle stepped with the same Philox actions, the tracker fed the oracle's outputs; tracking switched on
    before output `on_at` (-1: before the reset), every third env's reset scheduled before step `mask_at`.  Returns the
    tracker and the OR of the env flags seen."""
    from oracle.oracle import Oracle
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    g, ora = BatchedPredPreyGrass(cfg, n_envs), Oracle(cfg, n_envs, threads=8)
    tr = Tracker(n_envs, cfg.n_possible)
    flags = 0
    try:
        if on_at < 0:
            g.track_returns()
        g.reset()
        out = ora.reset()
        if on_at < 0:
            tr.update(out)
            _compare(g, tr, out["n"], "reset")
        for t in range(steps):
            if t == on_at:
                g.track_returns()
                tr.invalidate()
            if t == mask_at:
                mask = (np.arange(n_envs) % 3 == 0).astype(np.uint8)
                g.reset(mask=mask)
                ora.reset(mask=mask)
            a0, a1 = g.random_actions(action_seed)
            o0, o1 = ora.random_actions(action_seed)
            g.step(a0, a1)
            out = ora.step(_padded(o0), _padded(o1))
            flags |= int(np.bitwise_or.reduce(out["env_flags"]))
            if t >= on_at:
                tr.update(out)
                if t % every == 0 or t == steps - 1:
                    _compare(g, tr, out["n"], f"step {t}")
        # the aggregate: counts, max and -min exact, sums to 1e-12 (numpy sums in its own order)
        got, want = g.episode_stats_device().cpu().numpy(), tr.stats()
        counts = [0, 1, 8, 9, 11, 12, 13, 15]
        assert np.array_equal(got[counts], want[counts]) and np.array_equal(got[6:8], want[6:8]), (got, want)
        assert np.allclose(got, want, rtol=1e-12, atol=0.0), (got, want)
        return tr, flags
    finally:
        g.close()
        ora.close()


# ------------------------------------------------------------------------------------------------ bit-exact against the tracker
def test_returns_base_4096_envs_truncation_and_extinction():
    tr, flags = _lockstep(make_config(dict(BASE_CONFIG, max_steps=45), cap_live=(64, 192), seed=11), 4096, 100)
    assert flags & 1 and flags & 2  # episodes end by extinction and by truncation
    assert tr.env_acc[:, 0].sum() >= 4096 * 2 and tr.env_acc[:, 9].sum() > 0 and tr.env_acc[:, 13].sum() > 0


def test_returns_add():
    _lockstep(make_config(dict(BASE_CONFIG, max_steps=30), reward_mode="additive", cap_live=(64, 192), seed=3), 512, 70)


@pytest.mark.parametrize("case", ["crowded", "id_pool_exhausted"])
def test_returns_eco(case):
    cfg = CONSERVATION_CASES["eco_crowded"]() if case == "crowded" else REUSE_CONFIG()
    tr, _ = _lockstep(cfg, 256, 90)
    assert tr.reused == 0 and tr.env_acc[:, 0].sum() > 0


@pytest.mark.parametrize("case", ["stag", "stag_not_strict"])
def test_returns_stag(case):
    tr, _ = _lockstep(CONSERVATION_CASES[case](), 512, 90)
    assert tr.env_acc[:, 0].sum() >= 512


@pytest.mark.parametrize("trait", ["metabolic", "investment", "cooperation", "cadence"])
def test_returns_trait_variants(trait):
    from predpreygrass_b200.config import TRAIT_CONFIGS

    _lockstep(make_config(dict(TRAIT_CONFIGS[trait], max_steps=50), variant=VARIANT_ECO, cap_live=(64, 160), seed=7), 256, 90)


# ------------------------------------------------------------------------------------------------ aggregate
def test_episode_stats_bit_identical_across_runs():
    import torch

    from predpreygrass_b200.batched import BatchedPredPreyGrass

    cfg = make_config(dict(BASE_CONFIG, max_steps=15), reward_mode="additive", cap_live=(64, 192), seed=4)
    vecs = []
    for _ in range(2):
        g = BatchedPredPreyGrass(cfg, 3000)
        g.track_returns()
        g.reset()
        for _ in range(40):
            g.step(*g.random_actions(8))
        vecs.append(g.episode_stats_device().clone())
        assert g.episode_stats_device().equal(vecs[-1])
        m = g.episode_metrics()
        assert m["num_episodes"] == int(vecs[-1][0]) > 3000 and np.isfinite(m["episode_return_mean"])
        g.episode_stats_clear()
        v = g.episode_stats_device().cpu().numpy()
        assert (v[:6] == 0).all() and (v[8:] == 0).all() and (v[6:8] == -np.inf).all()
        g.close()
    assert torch.equal(vecs[0].view(torch.int64), vecs[1].view(torch.int64))


# ------------------------------------------------------------------------------------------------ lifecycle
def test_masked_reset_abandons_the_episode():
    tr, flags = _lockstep(make_config(dict(BASE_CONFIG, max_steps=40), cap_live=(64, 192), seed=5), 256, 30, mask_at=10)
    assert flags & 4
    tr, _ = _lockstep(make_config(dict(ECO_CONFIG, max_steps=40), variant=VARIANT_ECO, cap_live=(64, 128), seed=5), 128, 30, mask_at=12)


def test_switch_on_mid_run():
    """envs become valid at their next reset; before that their rows carry NaN / 0"""
    tr, _ = _lockstep(make_config(dict(BASE_CONFIG, max_steps=12), cap_live=(64, 192), seed=6), 512, 40, on_at=5)
    assert (tr.env_valid == 1).all()


def test_snapshot_restore_and_error_state():
    from oracle.oracle import Oracle
    from predpreygrass_b200._lib import PpgError
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    cfg = make_config(dict(STAG_CONFIG, max_steps=25), variant=VARIANT_STAG, cap_live=(64, 192), seed=12)
    B = 256
    g, ora = BatchedPredPreyGrass(cfg, B), Oracle(cfg, B, threads=8)
    with pytest.raises(PpgError, match="tracking is off"):
        g.returns()
    with pytest.raises(PpgError, match="never switched on"):
        g.episode_stats_device()
    with pytest.raises(PpgError, match="never switched on"):
        g.episode_stats_clear()
    size_off = g.snapshot().size
    g.track_returns()
    tr = Tracker(B, cfg.n_possible)
    g.reset()
    tr.update(ora.reset())
    blob, first_actions = None, []
    for t in range(45):
        if t == 10:
            blob = g.snapshot()
            assert blob.size == size_off
        if t == 20:  # back to the state of step 10 on both sides: every env invalid until its next reset
            g.restore(blob)
            tr.invalidate()
            assert int(g.returns().env_valid.sum()) == 0 and bool(g.returns().env_return.isnan().all())
            ora.close()
            ora = Oracle(cfg, B, threads=8)
            ora.reset()
            for a in first_actions:
                ora.step(*a)
        a0, a1 = g.random_actions(3)
        o0, o1 = ora.random_actions(3)
        if t < 10:
            first_actions.append((_padded(o0), _padded(o1)))
        g.step(a0, a1)
        out = ora.step(_padded(o0), _padded(o1))
        tr.update(out)
        _compare(g, tr, out["n"], f"step {t}")
    assert (tr.env_valid == 1).all()  # every env reset since the restore
    g.track_returns(False)
    with pytest.raises(PpgError, match="tracking is off"):
        g.returns()
    g.episode_stats_device()  # the accumulators outlive switching off
    g.close()
    ora.close()


def test_step_host():
    from oracle.oracle import Oracle
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    cfg = make_config(dict(BASE_CONFIG, max_steps=15), cap_live=(64, 192), seed=2)
    B = 128
    g, ora = BatchedPredPreyGrass(cfg, B), Oracle(cfg, B, threads=8)
    host = g.make_host_buffers()
    g.track_returns()
    tr = Tracker(B, cfg.n_possible)
    g.reset()
    tr.update(ora.reset())
    for t in range(30):
        o0, o1 = ora.random_actions(5)
        host["actions0"][: len(o0)] = torch_from(o0)
        host["actions1"][: len(o1)] = torch_from(o1)
        g.step_host(host)
        out = ora.step(_padded(o0), _padded(o1))
        tr.update(out)
        _compare(g, tr, out["n"], f"step_host {t}")
    g.close()
    ora.close()


def torch_from(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a, np.int32))


# ------------------------------------------------------------------------------------------------ queued rollouts
@pytest.mark.parametrize("variant,groups,chain", [("base", 1, 0), ("base", 2, 0), ("base", 1, 1), ("eco", 1, 1), ("stag", 2, 0)])
def test_rollout_random_queued(variant, groups, chain):
    """55 steps of ppg_rollout_random in one call, no host synchronisation: the tracking state after them equals the
    tracker fed the oracle's 55 outputs, stepped one at a time"""
    import torch

    from oracle.oracle import Oracle
    from predpreygrass_b200 import _lib
    from predpreygrass_b200.pipelined import PipelinedPredPreyGrass
    from tests.test_gpu_rollout import _factory

    B, K, seed = 768, 55, 4321
    factory = _factory(variant)
    L = _lib.load()
    pipe = PipelinedPredPreyGrass(factory, B, groups=groups)
    before = L.ppg_set_pdl_chain(chain)
    try:
        for e in pipe.envs:
            e.track_returns()
        torch.cuda.synchronize()
        pipe.reset()
        pipe.rollout_random(K, seed)
        torch.cuda.synchronize()
        per = B // groups
        for gi, e in enumerate(pipe.envs):
            cfg = factory(gi * per)
            ora = Oracle(cfg, per, threads=8)
            tr = Tracker(per, cfg.n_possible)
            try:
                tr.update(ora.reset(None))
                for _ in range(K):
                    o0, o1 = ora.random_actions(seed)
                    out = ora.step(_padded(o0), _padded(o1))
                    tr.update(out)
                _compare(e, tr, out["n"], f"{variant} group {gi} chain {chain}")
                assert tr.env_acc[:, 0].sum() >= per
            finally:
                ora.close()
    finally:
        L.ppg_set_pdl_chain(before)
        pipe.close()


# ------------------------------------------------------------------------------------------------ non-interference, sharding
def test_tracking_changes_no_output_and_no_launch_when_off():
    from predpreygrass_b200.batched import BatchedPredPreyGrass
    from tests.parity import compare_outputs

    cfg = make_config(dict(ECO_CONFIG, max_steps=30), variant=VARIANT_ECO, cap_live=(64, 128), seed=8)
    a, b, c = BatchedPredPreyGrass(cfg, 256), BatchedPredPreyGrass(cfg, 256), BatchedPredPreyGrass(cfg, 256)
    a.track_returns()
    c.track_returns()
    c.track_returns(False)  # switched on and off again: allocated, but nothing launched
    for h in (a, b, c):
        h.reset()
    per_step = {}
    for t in range(50):
        for name, h in (("a", a), ("b", b), ("c", c)):
            n0 = h.launch_count()
            h.step(*h.random_actions(9))
            per_step.setdefault(name, set()).add(h.launch_count() - n0)
        compare_outputs(a.outputs_numpy(), b.outputs_numpy(), f"step {t}")
        compare_outputs(c.outputs_numpy(), b.outputs_numpy(), f"step {t}")
    assert per_step["b"] == per_step["c"] and len(per_step["b"]) == 1
    assert per_step["a"] == {next(iter(per_step["b"])) + 1}
    for h in (a, b, c):
        h.close()


def test_sharded_handles_equal_one_handle():
    import torch

    from predpreygrass_b200.batched import BatchedPredPreyGrass

    mk = lambda base: make_config(dict(BASE_CONFIG, max_steps=20), variant=VARIANT_BASE, cap_live=(64, 192), seed=10,  # noqa: E731
                                  env_index_base=base)
    B, lo = 600, 250
    one, parts = BatchedPredPreyGrass(mk(0), B), [BatchedPredPreyGrass(mk(0), lo), BatchedPredPreyGrass(mk(lo), B - lo)]
    for h in [one] + parts:
        h.track_returns()
        h.reset()
    for _ in range(45):
        for h in [one] + parts:
            h.step(*h.random_actions(17))
    r1, rp = one.returns(), [p.returns() for p in parts]
    for k in ("env_return", "env_valid", "env_acc"):
        whole = getattr(r1, k)
        split = torch.cat([getattr(r, k) for r in rp])
        assert torch.equal(whole.view(torch.uint8), split.view(torch.uint8)), k
    n1, ns = one.out.n_rows.tolist(), [p.out.n_rows.tolist() for p in parts]
    for s in range(2):  # rows: the old rows of all envs, then their newborn rows
        for k in ("row_return", "row_life"):
            col, cols = getattr(r1, k)[s], [getattr(r, k)[s] for r in rp]
            whole = col[: n1[s] + n1[2 + s]]
            split = torch.cat([c[: n[s]] for c, n in zip(cols, ns)] + [c[n[s]: n[s] + n[2 + s]] for c, n in zip(cols, ns)])
            assert torch.equal(whole.view(torch.uint8), split.view(torch.uint8)), (k, s)
    for h in [one] + parts:
        h.close()
