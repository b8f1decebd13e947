"""The per-environment entry points of the C ABI (snapshots, task blocks, debug dumps) take the environment index from the caller: indices
outside the real environments are refused before any copy.  A padding environment (the step kernel works on whole blocks) is frozen by
dm_create, and a snapshot written into it would revive it; an index past the padding would address a neighbouring buffer."""
import numpy as np
import pytest

from deepmimic_b200 import capi

pytestmark = pytest.mark.gpu

N = 33                                                                 # not a multiple of the launch quantum: the handle has padding environments
HUMANOID = ["--arg_file", "args/train_humanoid3d_spinkick_args.txt"]
TARGET = ["--motion_file", "data/datasets/test_clips_mini.txt", "--arg_file", "args/train_amp_target_humanoid3d_locomotion_args.txt"]


def _steps(core):
    import torch
    A, S = core.dims.action_size, core.dims.state_size
    off = torch.tensor(core.static(capi.DM_ACTION_OFFSET), dtype=torch.float32, device="cuda")
    core.set_action((-off).expand(N, A).contiguous())
    core.update(1.0 / 600.0, 20)
    obs, rew = torch.zeros(N, S, device="cuda"), torch.zeros(N, device="cuda")
    core.observe(obs, rew)
    core.sync()
    assert torch.isfinite(obs).all() and torch.isfinite(rew).all()
    assert core.counters()[1] == 0


def test_out_of_range_environment_indices_are_refused(asset_root):
    core = capi.BatchedCore(HUMANOID, N, asset_root, seed=4)
    assert core.plan_launch(N)["padded_envs"] > N
    snap = core.get_snapshot(N - 1)
    core.debug_enable(True)
    for env in (N, -1):
        with pytest.raises(RuntimeError, match="dm_get_snapshot: environment %d" % env):
            core.get_snapshot(env)
        with pytest.raises(RuntimeError, match="dm_set_snapshot: environment %d" % env):
            core.set_snapshot(env, snap)
        with pytest.raises(RuntimeError, match="dm_get_debug: environment %d" % env):
            core.get_debug(env)
    core.debug_enable(False)
    core.set_snapshot(N - 1, snap)
    np.testing.assert_allclose(core.get_snapshot(N - 1), snap, rtol=0, atol=1e-6)   # PD targets pass through a float rotation
    _steps(core)
    core.close()


def test_out_of_range_task_blocks_are_refused(asset_root):
    core = capi.BatchedCore(TARGET, N, asset_root, seed=4)
    assert core.plan_launch(N)["padded_envs"] > N
    block = core.task_state(N - 1)
    for env in (N, -1):
        with pytest.raises(RuntimeError, match="dm_get_task_state: environment %d" % env):
            core.task_state(env)
        with pytest.raises(RuntimeError, match="dm_set_task_state: environment %d" % env):
            core.set_task_state(env, block)
    core.set_task_state(N - 1, block)
    np.testing.assert_array_equal(core.task_state(N - 1), block)
    _steps(core)
    core.close()
