"""Agent state aligned with the rows (include/ppg.h ppg_agent_state) on the CPU: a numpy reference that builds every column
from one output and the per-env readers (`read_env`, `read_env_eco`, `read_env_stag`, `read_env_acc`), following the header's
semantics literally; run on the C oracle's outputs, where it must show the properties the semantics promise.  Also the ctypes
layout of the argument struct against the header and the SASS of the kernel.  tests/test_gpu_agent_state.py compares the
device with this reference bit for bit."""
import ctypes as C
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from predpreygrass_b200.config import (BASE_CONFIG, ROW_CARCASS, STAG_CONFIG, TRAIT_CADENCE, TRAIT_CONFIGS, VARIANT_BASE,
                                       VARIANT_ECO, VARIANT_STAG, PpgAgentStateArgs, make_config)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TERM, TRUNC, NEWBORN = 0x01, 0x02, 0x04
ENV_ENDED = 0x03
NAN = np.float64("nan")
# per-species columns: (dtype, sentinel of an absent row, trailing shape)
COLUMNS = {"present": (np.uint8, 0, ()), "pos": (np.int32, -1, (2,)), "energy": (np.float64, NAN, ()), "age": (np.int32, -1, ()),
           "trait": (np.float64, NAN, ()), "facing": (np.int8, -1, ()), "acc": (np.float64, NAN, ())}


def columns_of(cfg):
    """{column: (pred, prey) booleans}: the per-species columns the variant has (include/ppg.h ppg_agent_state)"""
    eco, stag = cfg.variant == VARIANT_ECO, cfg.variant == VARIANT_STAG
    cad = eco and cfg.trait_mode == TRAIT_CADENCE
    return {"present": (True, True), "pos": (True, True), "energy": (True, True), "age": (eco or stag, eco or stag),
            "trait": (eco or stag, eco), "facing": (stag, False), "acc": (cad, cad)}


def reader(src, cfg):
    """per-env reader over an object with the read_env* methods of the oracle (or BatchedPredPreyGrass): env -> dict with
    ids, xy, energy and the variant's age, trait, facing, acc as (pred, prey) pairs in the order of ids, plus the grass"""
    def read(e):
        if cfg.variant == VARIANT_ECO:
            st = src.read_env_eco(e)
            st["trait"] = st["speed"]
            if cfg.trait_mode == TRAIT_CADENCE:
                st["acc"] = src.read_env_acc(e)
        elif cfg.variant == VARIANT_STAG:
            st = src.read_env_stag(e)
            st["trait"] = (st["trait"], None)
            st["facing"] = (st["facing"], None)
        else:
            st = src.read_env(e)
        return st
    return read


def agent_state_reference(out, read_env, cfg, envs=None):
    """The columns of one output, per the semantics of include/ppg.h: row r of species s is present when its env's flags
    have neither TERMINATED nor TRUNCATED and read_env(row_env[r]) lists its id; its columns are that entry's, the other
    rows get the sentinels.  envs: the envs to evaluate (default all); rows of the others are reported in `checked`
    as False and hold sentinels.  -> dict: f"{col}{s}" [n_s] for the columns the variant has, checked{s}, grass_pos
    [B, n_grass, 2], grass_energy [B, n_grass], checked_envs (sorted array)"""
    B, ng = len(out["env_flags"]), cfg.n_grass
    envs = np.arange(B) if envs is None else np.unique(np.asarray(envs, np.int64))
    cols = columns_of(cfg)
    ref = {"checked_envs": envs, "grass_pos": np.full((B, ng, 2), -1, np.int32), "grass_energy": np.full((B, ng), NAN)}
    rows_of = []
    for s in range(2):
        n = out["n"][s]
        for c, (dt, sent, tail) in COLUMNS.items():
            if cols[c][s]:
                ref[f"{c}{s}"] = np.full((n,) + tail, sent, dt)
        row_env = out[f"row_env{s}"][:n]
        order = np.argsort(row_env, kind="stable")
        bounds = np.searchsorted(row_env[order], np.arange(B + 1))
        rows_of.append((order, bounds))
        ref[f"checked{s}"] = np.isin(row_env, envs)
    for e in envs:
        if out["env_flags"][e] & ENV_ENDED:
            continue
        st = read_env(int(e))
        ref["grass_pos"][e] = st["grass_xy"][:ng]
        ref["grass_energy"][e] = st["grass_energy"][:ng]
        for s in range(2):
            order, bounds = rows_of[s]
            rows = order[bounds[e]: bounds[e + 1]]
            ids = np.asarray(st["ids"][s])
            if len(rows) == 0 or len(ids) == 0:
                continue
            srt = np.argsort(ids, kind="stable")
            rid = out[f"row_agent{s}"][rows]
            k = np.minimum(np.searchsorted(ids[srt], rid), len(ids) - 1)
            hit = ids[srt][k] == rid
            r, i = rows[hit], srt[k[hit]]
            ref[f"present{s}"][r] = 1
            ref[f"pos{s}"][r] = np.asarray(st["xy"][s])[i]
            ref[f"energy{s}"][r] = np.asarray(st["energy"][s])[i]
            for c in ("age", "trait", "facing", "acc"):
                if cols[c][s]:
                    ref[f"{c}{s}"][r] = np.asarray(st[c][s])[i]
    return ref


# ------------------------------------------------------------------------------------------------ the reference on the oracle
def _eco_carcasses():
    from tests.test_gpu_parity_eco import CROWDED

    return dict(CROWDED, max_energy_gain_per_prey=0.8, max_energy_gain_per_grass=1.0)


CASES = {
    "base": lambda: make_config(dict(BASE_CONFIG, max_steps=25), cap_live=(64, 192), seed=3),
    "base_extinction": lambda: make_config(dict(BASE_CONFIG, max_steps=100, n_initial_active_predator=2, n_initial_active_prey=3),
                                           cap_live=(64, 192), seed=3),
    "eco_carcasses": lambda: make_config(dict(_eco_carcasses(), max_steps=60), variant=VARIANT_ECO, cap_live=(64, 64), seed=9),
    "metabolic": lambda: make_config(dict(TRAIT_CONFIGS["metabolic"], max_steps=50), variant=VARIANT_ECO, cap_live=(64, 160), seed=7),
    "investment": lambda: make_config(dict(TRAIT_CONFIGS["investment"], max_steps=50), variant=VARIANT_ECO, cap_live=(64, 160), seed=7),
    "cooperation": lambda: make_config(dict(TRAIT_CONFIGS["cooperation"], max_steps=50), variant=VARIANT_ECO, cap_live=(64, 160), seed=7),
    "cadence": lambda: make_config(dict(TRAIT_CONFIGS["cadence"], max_steps=50), variant=VARIANT_ECO, cap_live=(64, 160), seed=7),
    "stag_strict": lambda: make_config(dict(STAG_CONFIG, max_steps=40), variant=VARIANT_STAG, cap_live=(64, 192), seed=6),
    "stag_not_strict": lambda: make_config(dict(STAG_CONFIG, max_steps=40, strict_rllib_output=False), variant=VARIANT_STAG,
                                           cap_live=(64, 192), seed=6),
}


def check_properties(out, ref, read_env, cfg, where):
    """the properties the semantics promise, on one output -> counts (present rows, ECO carcass rows present)"""
    counts = np.zeros(2, np.int64)
    ef = out["env_flags"]
    for s in range(2):
        n = out["n"][s]
        f, env = out[f"flags{s}"][:n], out[f"row_env{s}"][:n]
        pres = ref[f"present{s}"] == 1
        cont = (ef[env] & ENV_ENDED) == 0
        assert not pres[~cont].any(), where  # every row of an ended env is absent
        live = cont & ((f & (TERM | TRUNC)) == 0)
        assert pres[live].all(), where  # in an env that continues, every row flagged neither TERMINATED nor TRUNCATED is present
        term = cont & ((f & TERM) != 0)
        if cfg.variant == VARIANT_ECO:
            if s == 1:
                assert np.array_equal(pres[term], (f[term] & ROW_CARCASS) != 0), where  # a carcass stays in the list
            counts[1] += int((pres & ((f & ROW_CARCASS) != 0)).sum())
        else:
            assert not pres[term].any(), where  # BASE and STAG deaths leave the list
        counts[0] += int(pres.sum())
        # sentinels where absent
        assert (ref[f"pos{s}"][~pres] == -1).all() and np.isnan(ref[f"energy{s}"][~pres]).all(), where
        assert (ref[f"pos{s}"][pres] >= 0).all() and not np.isnan(ref[f"energy{s}"][pres]).any(), where
    # present rows plus list entries without a row equal the list lengths
    for e in np.nonzero((ef & ENV_ENDED) == 0)[0][:8]:
        st = read_env(int(e))
        for s in range(2):
            n = out["n"][s]
            env, ids = out[f"row_env{s}"][:n], out[f"row_agent{s}"][:n]
            mine = env == e
            listed = np.asarray(st["ids"][s])
            without_row = int((~np.isin(listed, ids[mine])).sum())
            assert int(ref[f"present{s}"][mine].sum()) + without_row == len(listed), (where, e, s)
    return counts


@pytest.mark.parametrize("case", sorted(CASES))
def test_reference_properties_on_the_oracle(case):
    from oracle.oracle import Oracle

    cfg = CASES[case]()
    B, T = 32, 90
    ora = Oracle(cfg, B, threads=4)
    read = reader(ora, cfg)
    totals, flags, ends_with_births = np.zeros(2, np.int64), 0, 0
    try:
        out = ora.reset()
        for t in range(T + 1):
            ref = agent_state_reference(out, read, cfg)
            totals += check_properties(out, ref, read, cfg, f"{case} output {t}")
            ef = out["env_flags"]
            flags |= int(np.bitwise_or.reduce(ef))
            ends_with_births += int((((ef & ENV_ENDED) != 0) & ((out["new_cnt0"] + out["new_cnt1"]) > 0)).sum())
            for e in np.nonzero(ef & ENV_ENDED)[0]:  # grass of an ended env: sentinels
                assert (ref["grass_pos"][e] == -1).all() and np.isnan(ref["grass_energy"][e]).all()
            if t == T:
                break
            a0, a1 = ora.random_actions(7)
            A0 = np.zeros(max(1, len(a0)), np.int32); A0[: len(a0)] = a0
            A1 = np.zeros(max(1, len(a1)), np.int32); A1[: len(a1)] = a1
            out = ora.step(A0, A1)
    finally:
        ora.close()
    assert totals[0] > 1000, totals
    assert flags & ENV_ENDED, case  # episodes end inside the run
    if case == "eco_carcasses":
        assert totals[1] > 0 and ends_with_births > 0  # carcass rows are present; episodes end on steps with births
    if case == "base_extinction":
        assert flags & 1


def test_reference_sentinels_and_subsets():
    """envs outside the evaluated subset are not read and keep the sentinels; the subset's rows equal the full evaluation"""
    from oracle.oracle import Oracle

    cfg = CASES["stag_strict"]()
    ora = Oracle(cfg, 12, threads=2)
    try:
        out = ora.reset()
        for _ in range(5):
            a0, a1 = ora.random_actions(3)
            out = ora.step(np.append(a0, 0).astype(np.int32), np.append(a1, 0).astype(np.int32))
        read = reader(ora, cfg)
        full = agent_state_reference(out, read, cfg)
        seen = []
        part = agent_state_reference(out, lambda e: seen.append(e) or read(e), cfg, envs=[1, 5])
        assert sorted(set(seen)) == [e for e in (1, 5) if not out["env_flags"][e] & ENV_ENDED]
        for s in range(2):
            k = part[f"checked{s}"]
            assert k.any() and not k.all()
            for c in ("present", "pos", "energy", "age"):
                assert np.array_equal(part[f"{c}{s}"][k], full[f"{c}{s}"][k])
            assert (part[f"present{s}"][~k] == 0).all()
        assert "facing1" not in full and "trait1" not in full and "acc0" not in full
    finally:
        ora.close()


# ------------------------------------------------------------------------------------------------ C-ABI
def _header_struct(name):
    hdr = open(os.path.join(ROOT, "include", "ppg.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), hdr, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    return re.findall(r"^\s*([a-z0-9_]+)\s*\*\s*([a-z_]+)(\[2\])?;", body, re.M)


def test_args_struct_matches_the_header():
    fields = _header_struct("ppg_agent_state_args")
    assert [f[1] for f in fields] == [f for f, _ in PpgAgentStateArgs._fields_]
    for (ctype, name, arr), (pname, ptype) in zip(fields, PpgAgentStateArgs._fields_):
        assert C.sizeof(ptype) == C.sizeof(C.c_void_p) * (2 if arr else 1), name
    assert C.sizeof(PpgAgentStateArgs) == 16 * C.sizeof(C.c_void_p)
    # the Python columns and dtypes follow the header's element types
    elem = {f[1]: f[0] for f in fields}
    want = {"uint8_t": np.uint8, "int32_t": np.int32, "double": np.float64, "int8_t": np.int8}
    for c, (dt, _, _) in COLUMNS.items():
        assert want[elem[c]] == dt, c


def test_python_columns_match_the_reference():
    pytest.importorskip("torch")
    from predpreygrass_b200.batched import AGENT_STATE_COLUMNS, agent_state_columns

    assert list(AGENT_STATE_COLUMNS) == list(COLUMNS)
    for case in ("base", "cadence", "metabolic", "stag_strict"):
        assert agent_state_columns(CASES[case]()) == columns_of(CASES[case]())
    assert columns_of(CASES["base"]())["age"] == (False, False) and CASES["base"]().variant == VARIANT_BASE


def test_agent_state_null_handle_is_invalid():
    from predpreygrass_b200 import _lib
    from predpreygrass_b200.build import build

    build()
    assert _lib.load().ppg_agent_state(None, None, None) == 1  # PPG_ERR_INVALID


CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


@pytest.mark.skipif(not os.path.exists(CUOBJDUMP), reason="cuobjdump not available")
def test_agent_state_kernel_never_triggers_dependent_launches():
    """ppg_agent_state is a plain launch after the observation kernel: it must not execute griddepcontrol.launch_dependents
    (PREEXIT) or wait on one (ACQBULK), or with the launch chain on the next step could rewrite the lists and rows it reads"""
    from predpreygrass_b200 import _lib
    from predpreygrass_b200.build import build

    build()
    sass = subprocess.run([CUOBJDUMP, "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    funcs = {m.group(1): body for m, body in zip(re.finditer(r"Function : (\S+)", sass), re.split(r"Function : \S+", sass)[1:])}
    mine = {f: b for f, b in funcs.items() if "ppg_agent_state_kernel" in f}
    assert len(mine) == 1, sorted(mine)
    for f, body in mine.items():
        assert "STG" in body and "PREEXIT" not in body and "ACQBULK" not in body, f
