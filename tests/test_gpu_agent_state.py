"""Agent state aligned with the rows on the GPU (`-m gpu`, include/ppg.h ppg_agent_state): every column of the device equals,
bit for bit, the numpy reference of tests/test_agent_state_cpu.py fed the oracle's outputs and the oracle's per-env readers,
with the oracle stepped in lockstep.  Also queued steps with the launch chain off and on, ppg_rollout_random, ppg_step_host,
the one-kernel step, non-interference with the outputs and the launch count, and the error paths."""
import numpy as np
import pytest

from predpreygrass_b200.config import (BASE_CONFIG, ECO_CONFIG, ROW_CARCASS, STAG_CONFIG, TRAIT_CONFIGS, VARIANT_ECO, VARIANT_STAG,
                                       make_config)
from tests.test_agent_state_cpu import COLUMNS, _eco_carcasses, agent_state_reference, columns_of, reader

pytestmark = pytest.mark.gpu

ENV_ENDED, ENV_TERM, ENV_TRUNC, ENV_RESET, ENV_IDLE = 0x03, 0x01, 0x02, 0x04, 0x08


def _padded(a):
    A = np.zeros(max(1, len(a)), np.int32)
    A[: len(a)] = a
    return A


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64) if a.dtype == np.float64 else a


def compare_state(st, ref, cfg, n, where):
    """the device's AgentState against the reference on the reference's checked rows and envs, bit for bit (NaN included)"""
    cols = columns_of(cfg)
    for s in range(2):
        k = ref[f"checked{s}"]
        for c in COLUMNS:
            t = getattr(st, c)[s]
            if not cols[c][s]:
                assert t is None, (where, c, s)
                continue
            got, want = t[: n[s]].cpu().numpy(), ref[f"{c}{s}"]
            assert got.dtype == want.dtype, (where, c, s)
            g, w = _bits(got[k]), _bits(want[k])
            if not np.array_equal(g, w):
                bad = np.nonzero((g != w).reshape(len(g), -1).any(axis=1))[0][:5]
                raise AssertionError(f"{where}: {c}{s} differs at checked rows {bad.tolist()}: gpu={got[k][bad].tolist()} "
                                     f"reference={want[k][bad].tolist()}")
    envs = ref["checked_envs"]
    assert np.array_equal(st.grass_pos.cpu().numpy()[envs], ref["grass_pos"][envs]), (where, "grass_pos")
    assert np.array_equal(_bits(st.grass_energy.cpu().numpy()[envs]), _bits(ref["grass_energy"][envs])), (where, "grass_energy")


def _clone(st):
    from dataclasses import fields, replace

    return replace(st, **{f.name: (tuple(None if t is None else t.clone() for t in getattr(st, f.name))
                                   if isinstance(getattr(st, f.name), tuple) else getattr(st, f.name).clone()) for f in fields(st)})


def _equal(a, b):
    from dataclasses import fields

    for f in fields(a):
        x, y = getattr(a, f.name), getattr(b, f.name)
        for u, v in (zip(x, y) if isinstance(x, tuple) else [(x, y)]):
            if (u is None) != (v is None) or (u is not None and not np.array_equal(_bits(u.cpu().numpy()), _bits(v.cpu().numpy()))):
                return False
    return True


def _lockstep(cfg, n_envs, steps, *, full_every=1, rotate=16, mask_at=None, action_seed=31):
    """GPU and oracle stepped with the same Philox actions.  After every output agent_state() is compared with the reference:
    on every env when t % full_every == 0, at the last output, on outputs where an episode is truncated and on the outputs
    right after them (which reset those envs), else on the envs e with e % rotate == t % rotate.  mask_at: before that step, every third env's reset is scheduled on both sides, and the
    call between the masked reset and the step must still describe the last output.  -> stats of what was seen"""
    import torch

    from oracle.oracle import Oracle
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    g, ora = BatchedPredPreyGrass(cfg, n_envs), Oracle(cfg, n_envs, threads=8)
    read = reader(ora, cfg)
    seen = {"flags": 0, "full": 0, "full_ends": 0, "full_resets": 0, "ends_with_births": 0, "carcass_rows": 0, "present": 0}
    prev_trunc = [False]

    def check(t, out):
        ef = out["env_flags"]
        trunc = bool((ef & ENV_TRUNC).any())
        full = t % full_every == 0 or t == steps or trunc or prev_trunc[0]
        prev_trunc[0] = trunc
        envs = None if full else np.nonzero(np.arange(n_envs) % rotate == t % rotate)[0]
        st = g.agent_state()
        ref = agent_state_reference(out, read, cfg, envs)
        for s in range(2):
            assert np.array_equal(g.out.row_agent[s][: out["n"][s]].cpu().numpy(), out[f"row_agent{s}"]), (t, s)
        compare_state(st, ref, cfg, out["n"], f"output {t}")
        seen["flags"] |= int(np.bitwise_or.reduce(ef))
        seen["full"] += full
        seen["full_ends"] += full and bool((ef & ENV_ENDED).any())
        seen["full_resets"] += full and t > 0 and bool((ef & ENV_RESET).any())
        seen["ends_with_births"] += int((((ef & ENV_ENDED) != 0) & ((out["new_cnt0"] + out["new_cnt1"]) > 0)).sum())
        for s in range(2):
            p = st.present[s][: out["n"][s]].cpu().numpy() == 1
            seen["present"] += int(p.sum())
            seen["carcass_rows"] += int((p & ((out[f"flags{s}"] & ROW_CARCASS) != 0)).sum())

    try:
        g.reset()
        check(0, ora.reset())
        for t in range(1, steps + 1):
            if t == mask_at:
                before = _clone(g.agent_state())
                mask = (np.arange(n_envs) % 3 == 0).astype(np.uint8)
                g.reset(mask=mask)
                ora.reset(mask=mask)
                assert _equal(g.agent_state(), before)  # a masked reset only schedules: still the last output
            a0, a1 = g.random_actions(action_seed)
            o0, o1 = ora.random_actions(action_seed)
            g.step(a0, a1)
            check(t, ora.step(_padded(o0), _padded(o1)))
        torch.cuda.synchronize()
        return seen
    finally:
        g.close()
        ora.close()


# ------------------------------------------------------------------------------------------------ bit-exact against the reference
def test_agent_state_base_4096_envs():
    seen = _lockstep(make_config(dict(BASE_CONFIG, max_steps=45), cap_live=(64, 192), seed=11), 4096, 80, full_every=8)
    assert seen["flags"] & ENV_TERM and seen["flags"] & ENV_TRUNC  # episodes end by extinction and by the time limit
    assert seen["full"] >= 10 and seen["full_ends"] >= 2 and seen["full_resets"] >= 2, seen


def test_agent_state_add():
    seen = _lockstep(make_config(dict(BASE_CONFIG, max_steps=30), reward_mode="additive", cap_live=(64, 192), seed=3), 512, 70)
    assert seen["flags"] & ENV_TRUNC


def test_agent_state_eco_carcasses_and_ghost_cells():
    ghost = dict(_eco_carcasses(), max_agent_age={"predator": None, "prey": 9}, max_energy_gain_per_prey=0.4, max_steps=40,
                 energy_gain_per_step_grass=0.8, prey_creation_energy_threshold=3.0)
    for cfg in (dict(_eco_carcasses(), max_steps=45), ghost):
        seen = _lockstep(make_config(cfg, variant=VARIANT_ECO, cap_live=(96, 192), seed=17), 256, 100)
        assert seen["carcass_rows"] > 0 and seen["ends_with_births"] > 0 and seen["flags"] & ENV_ENDED, seen


def test_agent_state_eco_id_pool_exhausted():
    from tests.test_returns_cpu import REUSE_CONFIG

    seen = _lockstep(REUSE_CONFIG(), 128, 100)
    assert seen["flags"] & ENV_TRUNC


@pytest.mark.parametrize("trait", ["metabolic", "investment", "cooperation", "cadence"])
def test_agent_state_trait_variants(trait):
    seen = _lockstep(make_config(dict(TRAIT_CONFIGS[trait], max_steps=50), variant=VARIANT_ECO, cap_live=(64, 160), seed=7), 256, 110)
    assert seen["flags"] & ENV_ENDED and seen["present"] > 0


def test_agent_state_stag_bench_caps_walls_and_not_strict():
    from tests.test_gpu_parity_stag import CROWDED

    cfg = make_config(dict(STAG_CONFIG, max_steps=60, n_initial_active_type_1_predator=2), variant=VARIANT_STAG, cap_live=(160, 640), seed=6)
    assert _lockstep(cfg, 512, 90, full_every=2)["flags"] & ENV_TRUNC
    walls = [(3, y) for y in range(2, 8)] + [(6, 1), (6, 2), (7, 7), (8, 7), (1, 8), (9, 9)]
    cfg = dict(CROWDED, grid_size=10, manual_wall_positions=walls, respect_los_for_movement=True, type_2_action_range=5, max_steps=50)
    assert _lockstep(make_config(cfg, variant=VARIANT_STAG, cap_live=(96, 224), seed=31), 256, 80)["flags"] & ENV_ENDED
    cfg = make_config(dict(STAG_CONFIG, max_steps=40, strict_rllib_output=False), variant=VARIANT_STAG, cap_live=(64, 192), seed=6)
    assert _lockstep(cfg, 256, 70)["flags"] & ENV_ENDED


def test_agent_state_masked_reset():
    assert _lockstep(make_config(dict(BASE_CONFIG, max_steps=40), cap_live=(64, 192), seed=5), 256, 30, mask_at=12)["flags"] & ENV_RESET
    cfg = make_config(dict(ECO_CONFIG, max_steps=40), variant=VARIANT_ECO, cap_live=(64, 128), seed=5)
    assert _lockstep(cfg, 128, 30, mask_at=9)["flags"] & ENV_RESET


def test_agent_state_autoreset_off_idle_envs():
    cfg = make_config(dict(BASE_CONFIG, max_steps=20), cap_live=(64, 192), seed=3, autoreset=False)
    assert _lockstep(cfg, 128, 40)["flags"] & ENV_IDLE
    cfg = make_config(dict(_eco_carcasses(), max_steps=30), variant=VARIANT_ECO, cap_live=(64, 64), seed=2, autoreset=False)
    assert _lockstep(cfg, 64, 50)["flags"] & ENV_IDLE


# ------------------------------------------------------------------------------------------------ other paths to an output
@pytest.mark.parametrize("chain", [0, 1])
def test_agent_state_queued_without_host_synchronisation(chain):
    """20 x {random actions, step, agent_state() cloned} on one stream, nothing synchronised in between; with the launch chain
    on, the next step's kernels must not rewrite the lists or the rows while the agent-state kernel still reads them"""
    import torch

    from oracle.oracle import Oracle
    from predpreygrass_b200 import _lib
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    cfg = make_config(dict(STAG_CONFIG, max_steps=12), variant=VARIANT_STAG, cap_live=(64, 192), seed=13)
    B, T, seed = 512, 20, 555
    before = _lib.load().ppg_set_pdl_chain(chain)
    try:
        g = BatchedPredPreyGrass(cfg, B)
        g.reset()
        torch.cuda.synchronize()
        states = []
        for _ in range(T):
            g.step(*g.random_actions(seed))
            states.append(_clone(g.agent_state()))
        torch.cuda.synchronize()
    finally:
        _lib.load().ppg_set_pdl_chain(before)
    ora = Oracle(cfg, B, threads=8)
    read = reader(ora, cfg)
    ora.reset()
    for t in range(T):
        o0, o1 = ora.random_actions(seed)
        out = ora.step(_padded(o0), _padded(o1))
        compare_state(states[t], agent_state_reference(out, read, cfg), cfg, out["n"], f"queued step {t} (chain {chain})")
    g.close()
    ora.close()


def test_agent_state_after_rollout_random_two_groups():
    import torch

    from oracle.oracle import Oracle
    from predpreygrass_b200.pipelined import PipelinedPredPreyGrass
    from tests.test_gpu_rollout import _factory

    B, K, seed = 768, 45, 4321
    factory = _factory("eco")
    pipe = PipelinedPredPreyGrass(factory, B, groups=2)
    try:
        pipe.reset()
        pipe.rollout_random(K, seed)
        torch.cuda.synchronize()  # the groups ran on their own streams; agent_state() runs on the current one
        states = [e.agent_state() for e in pipe.envs]
        torch.cuda.synchronize()
        per = B // 2
        for gi, st in enumerate(states):
            cfg = factory(gi * per)
            ora = Oracle(cfg, per, threads=8)
            try:
                ora.reset(None)
                for _ in range(K):
                    o0, o1 = ora.random_actions(seed)
                    out = ora.step(_padded(o0), _padded(o1))
                compare_state(st, agent_state_reference(out, reader(ora, cfg), cfg), cfg, out["n"], f"group {gi}")
            finally:
                ora.close()
    finally:
        pipe.close()


def test_agent_state_after_step_host():
    import torch

    from oracle.oracle import Oracle
    from predpreygrass_b200.batched import BatchedPredPreyGrass

    cfg = make_config(dict(BASE_CONFIG, max_steps=15), cap_live=(64, 192), seed=2)
    B = 128
    g, ora = BatchedPredPreyGrass(cfg, B), Oracle(cfg, B, threads=8)
    read = reader(ora, cfg)
    host = g.make_host_buffers()
    g.reset()
    ora.reset()
    for t in range(25):
        o0, o1 = ora.random_actions(5)
        host["actions0"][: len(o0)] = torch.from_numpy(np.ascontiguousarray(o0, np.int32))
        host["actions1"][: len(o1)] = torch.from_numpy(np.ascontiguousarray(o1, np.int32))
        g.step_host(host)
        out = ora.step(_padded(o0), _padded(o1))
        compare_state(g.agent_state(), agent_state_reference(out, read, cfg), cfg, out["n"], f"step_host {t}")
    g.close()
    ora.close()


def test_agent_state_one_kernel_step(monkeypatch):
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
    assert seen["flags"] & ENV_ENDED and seen["flags"] & ENV_RESET


# ------------------------------------------------------------------------------------------------ isolation and errors
def test_agent_state_changes_no_output():
    """twin handles, one calling agent_state() after every output: bit-identical outputs, one launch more per call"""
    from predpreygrass_b200.batched import BatchedPredPreyGrass
    from tests.parity import compare_outputs

    cfg = make_config(dict(_eco_carcasses(), max_steps=30), variant=VARIANT_ECO, cap_live=(64, 64), seed=8)
    a, b = BatchedPredPreyGrass(cfg, 256), BatchedPredPreyGrass(cfg, 256)
    a.reset(); b.reset()
    calls = 0
    for t in range(50):
        a.agent_state()
        calls += 1
        a.step(*a.random_actions(9))
        b.step(*b.random_actions(9))
        compare_outputs(a.outputs_numpy(), b.outputs_numpy(), f"step {t}")
    assert a.launch_count() - b.launch_count() == calls
    a.close(); b.close()


def test_agent_state_errors_and_out():
    import ctypes as C

    import torch

    from predpreygrass_b200 import _lib
    from predpreygrass_b200._lib import PpgError
    from predpreygrass_b200.batched import BatchedPredPreyGrass
    from predpreygrass_b200.config import PpgAgentStateArgs

    L = _lib.load()
    g = BatchedPredPreyGrass(make_config(BASE_CONFIG, cap_live=(64, 192), seed=1), 16)
    with pytest.raises(PpgError, match="no output since ppg_create"):
        g.agent_state()
    g.reset()
    g.step(*g.random_actions(1))
    blob = g.snapshot()
    st = g.new_agent_state()
    # rows at or beyond the output's row count are left untouched
    for s in range(2):
        st.present[s].fill_(0xAB)
        st.energy[s].fill_(7.0)
    assert g.agent_state(out=st) is st
    n = g.out.counts()
    for s in range(2):
        assert bool((st.present[s][n[s]:] == 0xAB).all()) and bool((st.energy[s][n[s]:] == 7.0).all())
        assert bool((st.present[s][: n[s]] <= 1).all())
    # a NULL column is not written
    keep = st.pos[0].clone()
    g.agent_state(out=type(st)(**{**st.__dict__, "pos": (None, st.pos[1])}))
    assert st.pos[0].equal(keep)
    # C-ABI: NULL present, a column the variant lacks
    a = PpgAgentStateArgs()
    a.present[0] = st.present[0].data_ptr()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert L.ppg_agent_state(g.h, C.byref(a), stream) == 1
    a.present[1] = st.present[1].data_ptr()
    assert L.ppg_agent_state(g.h, C.byref(a), stream) == 0
    age = torch.empty(g.row_capacity[0], dtype=torch.int32, device=g.device)
    a.age[0] = age.data_ptr()
    assert L.ppg_agent_state(g.h, C.byref(a), stream) == 1 and b"age" in L.ppg_last_error(g.h)
    # Python: a bad out raises ValueError
    cap = g.row_capacity
    bad = [("energy", (torch.empty(cap[0], dtype=torch.float32, device=g.device), st.energy[1])),
           ("energy", (torch.empty(cap[0] - 1, dtype=torch.float64, device=g.device), st.energy[1])),
           ("pos", (torch.empty((cap[0], 4), dtype=torch.int32, device=g.device)[:, ::2], st.pos[1])),
           ("present", (None, st.present[1])),
           ("age", (age, None)),
           ("energy", (torch.empty(cap[0], dtype=torch.float64), st.energy[1]))]
    for k, v in bad:
        with pytest.raises(ValueError):
            g.agent_state(out=type(st)(**{**st.__dict__, k: v}))
    with pytest.raises(ValueError):
        g.agent_state(out=type(st)(**{**st.__dict__, "grass_energy": torch.empty((16, 3), dtype=torch.float64, device=g.device)}))
    # after restore: no output until the next step
    g.restore(blob)
    with pytest.raises(PpgError, match="ppg_restore"):
        g.agent_state()
    g.step(*g.random_actions(1))
    g.agent_state()
    g.close()
    # variants: the columns each one has
    s = BatchedPredPreyGrass(make_config(STAG_CONFIG, variant=VARIANT_STAG, cap_live=(64, 160), seed=2), 4)
    s.reset()
    st = s.agent_state()
    assert st.facing[0].dtype == torch.int8 and st.facing[1] is None and st.trait[1] is None and st.acc == (None, None)
    a = PpgAgentStateArgs()
    a.present[0], a.present[1] = st.present[0].data_ptr(), st.present[1].data_ptr()
    a.facing[1] = st.present[1].data_ptr()
    assert L.ppg_agent_state(s.h, C.byref(a), stream) == 1 and b"facing" in L.ppg_last_error(s.h)
    a.facing[1] = None
    a.acc[0] = st.energy[0].data_ptr()
    assert L.ppg_agent_state(s.h, C.byref(a), stream) == 1 and b"acc" in L.ppg_last_error(s.h)
    s.close()
