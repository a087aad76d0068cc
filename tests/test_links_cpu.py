"""Row links between consecutive outputs (include/ppg.h ppg_track_links) on the CPU: a numpy reference of prev_row that follows
the header literally, run on the C oracle's outputs, where it must be the inverse of ppg_gae's successor links
(tests/test_gae_cpu.py's reference next_row); the two facts about the agent lists the kernel relies on; the ctypes mirror of
the C-ABI; and the SASS of the kernel.  tests/test_gpu_links.py compares the device with this reference bit for bit."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from predpreygrass_b200.config import VARIANT_ECO, make_config
from tests.test_gae_cpu import _case, gae_reference, oracle_rollout, synth_values

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TERM, TRUNC, NEWBORN, FOUNDER, CARCASS = 0x01, 0x02, 0x04, 0x08, 0x20
ENV_RESET = 0x04


def prev_rows(o0, o1):
    """prev_row of output o1 given the output o0 before it, per species int32 [n1]: an old row (r < n_old) not flagged
    FOUNDER, of an env whose output is not a reset, gets the row of the same (env, id) in o0; every other row -1"""
    res = []
    for s in range(2):
        n0, n1, n1_old = o0["n"][s], o1["n"][s], o1["n_old"][s]
        at = {(int(e), int(i)): r for r, (e, i) in enumerate(zip(o0[f"row_env{s}"][:n0], o0[f"row_agent{s}"][:n0]))}
        env, ids, f = o1[f"row_env{s}"][:n1], o1[f"row_agent{s}"][:n1], o1[f"flags{s}"][:n1]
        pr = np.full(n1, -1, np.int32)
        for r in range(n1_old):
            if not f[r] & FOUNDER and not o1["env_flags"][env[r]] & ENV_RESET:
                pr[r] = at[(int(env[r]), int(ids[r]))]  # KeyError: an old row without a row in the output before
        res.append(pr)
    return res


def _eco_carcass_case():
    from tests.test_agent_state_cpu import _eco_carcasses

    return make_config(dict(_eco_carcasses(), max_steps=45), variant=VARIANT_ECO, cap_live=(96, 192), seed=17), 64, 80, {}


CASES = ["base_truncation", "base_extinction", "eco_crowded", "eco_carcass", "eco_pool_exhausted", "stag_strict", "stag_not_strict",
         "base_masked_reset", "base_autoreset_off"]


def _rollout(case):
    cfg, B, T, kw = _eco_carcass_case() if case == "eco_carcass" else _case(case)
    return oracle_rollout(cfg, B, T, **kw)


@pytest.mark.parametrize("case", CASES)
def test_prev_row_is_the_inverse_of_next_row(case):
    outputs = _rollout(case)
    ref = gae_reference(outputs, [synth_values(o, t) for t, o in enumerate(outputs)], 0.9, 0.8)
    linked = 0
    for t in range(len(outputs) - 1):
        prev = prev_rows(outputs[t], outputs[t + 1])
        for s in range(2):
            nxt = ref[s]["next_row"][t]
            inv = np.full(outputs[t + 1]["n"][s], -1, np.int32)
            inv[nxt[nxt >= 0]] = np.nonzero(nxt >= 0)[0]
            assert np.array_equal(prev[s], inv), (case, t, s)
            linked += int((prev[s] >= 0).sum())
    assert linked > 1000, linked
    ef = np.bitwise_or.reduce([int(np.bitwise_or.reduce(o["env_flags"])) for o in outputs])
    if case == "base_masked_reset":
        assert ef & ENV_RESET
    if case == "base_autoreset_off":
        assert ef & 0x08  # idle envs


@pytest.mark.parametrize("case", CASES)
def test_list_facts_the_kernel_relies_on(case):
    """within an episode of an env no id is handed out twice (a NEWBORN row's id was never seen before in the episode), and
    the id of a TERMINATED row never shows up as an old row of a later output.  The latter covers the ECO carcass (a prey
    that died bitten but not fully eaten, flagged TERMINATED | CARCASS), which stays in its env's list with the stale row
    of its last output: that entry is never looked up"""
    outputs = _rollout(case)
    carcasses = 0
    for s in range(2):
        seen, dead = {}, {}
        for o in outputs:
            n, n_old = o["n"][s], o["n_old"][s]
            env, ids, f = o[f"row_env{s}"][:n], o[f"row_agent{s}"][:n], o[f"flags{s}"][:n]
            for e in np.nonzero(o["env_flags"] & ENV_RESET)[0]:
                seen[int(e)], dead[int(e)] = set(), set()
            for r in range(n):
                e, i = int(env[r]), int(ids[r])
                sset, dset = seen.setdefault(e, set()), dead.setdefault(e, set())
                if r < n_old and not f[r] & FOUNDER:
                    assert i not in dset, (case, s, e, i)
                if f[r] & NEWBORN:
                    assert i not in sset, (case, s, e, i)
                sset.add(i)
            for r in np.nonzero(f & TERM)[0]:
                dead[int(env[r])].add(int(ids[r]))
                carcasses += bool(f[r] & CARCASS)
    if case == "eco_carcass":
        assert carcasses > 0


# ------------------------------------------------------------------------------------------------ C-ABI
def _header():
    return open(os.path.join(ROOT, "include", "ppg.h")).read()


def test_ctypes_mirror_matches_the_header():
    from predpreygrass_b200 import _lib
    from predpreygrass_b200.config import LINK_ERR_MISSING, LINK_ERR_OVERFLOW

    hdr = _header()
    defs = dict(re.findall(r"#define (PPG_LINK_ERR_\w+) (0x[0-9a-f]+)u", hdr))
    assert {k: int(v, 16) for k, v in defs.items()} == {"PPG_LINK_ERR_MISSING": LINK_ERR_MISSING,
                                                         "PPG_LINK_ERR_OVERFLOW": LINK_ERR_OVERFLOW}
    protos = {m.group(1): m.group(2) for m in re.finditer(r"int (ppg_track_links|ppg_get_links)\(([^)]*)\);", hdr)}
    assert protos["ppg_track_links"].replace(" ", "") == "ppg_handleh,int32_ton,void*cuda_stream"
    assert protos["ppg_get_links"].replace(" ", "") == "ppg_handleh,int32_t**prev_row,uint32_t**error"
    assert "ppg_track_links" in _lib.SYMBOLS and "ppg_get_links" in _lib.SYMBOLS
    assert re.search(r"#define PPG_ABI_VERSION 10\b", hdr)


def test_python_binding_argtypes():
    import ctypes as C

    from predpreygrass_b200 import _lib
    from predpreygrass_b200.build import build

    build()
    L = _lib.load()
    assert L.ppg_track_links.argtypes == [C.c_void_p, C.c_int32, C.c_void_p]
    assert len(L.ppg_get_links.argtypes) == 3
    rows, err = (C.c_void_p * 2)(), C.c_void_p()
    assert L.ppg_get_links(None, C.byref(rows), C.byref(err)) == 1  # NULL handle: PPG_ERR_INVALID
    assert L.ppg_track_links(None, 1, None) == 1


CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


@pytest.mark.skipif(not os.path.exists(CUOBJDUMP), reason="cuobjdump not available")
def test_links_kernel_never_triggers_dependent_launches():
    """ppg_links_kernel is a plain launch after the observation kernel: it must not execute griddepcontrol.launch_dependents
    (PREEXIT) or wait on one (ACQBULK), or with the launch chain on the next step could rewrite the lists and rows it reads"""
    from predpreygrass_b200 import _lib
    from predpreygrass_b200.build import build

    build()
    sass = subprocess.run([CUOBJDUMP, "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    funcs = {m.group(1): body for m, body in zip(re.finditer(r"Function : (\S+)", sass), re.split(r"Function : \S+", sass)[1:])}
    mine = {f: b for f, b in funcs.items() if "ppg_links_kernel" in f}
    assert len(mine) == 1, sorted(mine)
    for f, body in mine.items():
        assert "STG" in body and "PREEXIT" not in body and "ACQBULK" not in body, f
