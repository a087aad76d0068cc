"""The world state in the CPU suite: the dict adapters' `grid_world_state` over the C oracle (tests/oracle_batch.py, extended
here by `world_state`) on the recorded episodes, the C-ABI's argument check, and a static guard on the SASS of
ppg_world_state_kernel."""
import os
import re
import shutil
import subprocess

import pytest

import predpreygrass_b200.batched as batched
from predpreygrass_b200 import _lib
from tests import test_gpu_world_state as W
from tests.helpers import golden_cases
from tests.oracle_batch import OracleBatch

CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


class OracleWorldBatch(OracleBatch):
    """OracleBatch plus `world_state` over the oracle's grid (`ppgo_read_grid`, float64, rounded to float32 like the device)"""

    def world_state(self, env_begin=0, n=None):
        import numpy as np
        import torch

        n = self.n_envs - env_begin if n is None else n
        return torch.from_numpy(np.stack([self.o.read_grid(e).astype(np.float32) for e in range(env_begin, env_begin + n)]))


@pytest.mark.parametrize("name", golden_cases(("eco", "stag", "mr", "inv", "coop", "cad")))
def test_adapter_grid_world_state_over_the_oracle(name, monkeypatch):
    monkeypatch.setattr(batched, "BatchedPredPreyGrass", OracleWorldBatch)
    W.replay_adapter_grid(name)


def test_world_state_null_handle_is_invalid():
    assert _lib.load().ppg_world_state(None, 0, 1, None, None) == 1  # PPG_ERR_INVALID


@pytest.mark.skipif(not os.path.exists(CUOBJDUMP), reason="cuobjdump not available")
def test_world_state_kernel_does_not_trigger_dependents():
    """With the launch chain on, the step kernel after ppg_world_state is launched with programmatic stream serialization:
    the world-state kernel must not execute griddepcontrol.launch_dependents (SASS `PREEXIT`), or that step kernel could
    overwrite the env images while they are still being read."""
    sass = subprocess.run([CUOBJDUMP, "-sass", _lib.LIB_PATH], capture_output=True, text=True, check=True).stdout
    fns = [f for f in re.split(r"Function : ", sass) if f.startswith("_ZN3ppg22ppg_world_state_kernel")]
    assert len(fns) == 2, len(fns)  # 8-bit and 16-bit owner maps
    assert all("STG" in f and "PREEXIT" not in f for f in fns)
