"""The fused env steps of Feeding, BedBathing, Dressing and ScratchItch share one driver in the C ABI: the same init check,
the same host-buffer and device-buffer paths, and the same NULL-`info` contract.  Runs on the kernel bodies compiled for
the host (tests/kernel_harness), where "device" buffers are host memory, so numpy arrays stand in for device tensors."""
import functools

import numpy as np
import pytest

from assistive_gym_b200 import capi
from assistive_gym_b200.bed_bathing_batch import BedBathingBatch
from assistive_gym_b200.dressing_batch import DressingBatch
from assistive_gym_b200.feeding_batch import FeedingBatch
from assistive_gym_b200.scratch_itch_batch import ScratchItchBatch
from assistive_gym_b200.sim import BatchSim, _p

N = 3
# task -> (batch class, ABI prefix, obs width, seeded reset)
TASKS = {
    'feeding': (FeedingBatch, 'feeding', 25, lambda b, sim: b.reset(sim, np.random.default_rng(1), settle_steps=5, impairment='tremor')),
    'bed_bathing': (BedBathingBatch, 'bathing', 24, lambda b, sim: b.reset(sim, np.random.default_rng(2))),
    'dressing': (DressingBatch, 'dressing', 24, lambda b, sim: b.reset(sim, np.random.default_rng(4), attempts=12, settle_steps=2)),
    'scratch_itch': (ScratchItchBatch, 'scratch', 30, lambda b, sim: b.reset(sim, np.random.default_rng(3))),
}


@functools.lru_cache(maxsize=None)
def _batch(task):
    return TASKS[task][0]()


def _sim(lib, task):
    b = _batch(task)
    cfg = DressingBatch.config() if task == 'dressing' else capi.default_config(residual_threshold=0.0)
    return BatchSim(b.scene, cfg, N, _lib=lib)


def _started(lib, task):
    """A sim after a seeded reset with the task's fused step armed: the same state every call."""
    b, reset = _batch(task), TASKS[task][3]
    sim = _sim(lib, task)
    b.start_fused(sim, reset(b, sim))
    return sim


def _outputs(obs_dim):
    return (np.zeros((N, obs_dim), dtype=np.float32), np.zeros(N, dtype=np.float32), np.zeros(N, dtype=np.float32),
            np.zeros((N, 4), dtype=np.float32))


def _actions(k):
    return np.random.default_rng(100 + k).uniform(-1.2, 1.2, size=(N, 7)).astype(np.float32)


@pytest.mark.parametrize('task', list(TASKS))
def test_step_before_init_raises(emu_lib, task):
    _, prefix, obs_dim, _ = TASKS[task]
    sim = _sim(emu_lib, task)
    a, out = _actions(0), _outputs(obs_dim)
    with pytest.raises(RuntimeError, match='ag_%s_init' % prefix):
        getattr(sim, prefix + '_step_host')(a)
    with pytest.raises(RuntimeError, match='ag_%s_init' % prefix):
        getattr(sim, prefix + '_step_dev')(a.ctypes.data, *[o.ctypes.data for o in out])
    sim.close()


@pytest.mark.parametrize('task', list(TASKS))
def test_step_dev_matches_step_host(emu_lib, task):
    _, prefix, obs_dim, _ = TASKS[task]
    host, dev = _started(emu_lib, task), _started(emu_lib, task)
    np.testing.assert_array_equal(host.state_get(), dev.state_get())
    for k in range(2):
        a = _actions(k)
        ref = getattr(host, prefix + '_step_host')(a)
        out = _outputs(obs_dim)
        getattr(dev, prefix + '_step_dev')(a.ctypes.data, *[o.ctypes.data for o in out])
        for x, y in zip(out, ref):
            np.testing.assert_array_equal(x, y)
    np.testing.assert_array_equal(host.state_get(), dev.state_get())
    host.close(), dev.close()


@pytest.mark.parametrize('task', list(TASKS))
def test_step_host_accepts_null_info(emu_lib, task):
    _, prefix, obs_dim, _ = TASKS[task]
    with_info, without = _started(emu_lib, task), _started(emu_lib, task)
    fn = getattr(emu_lib, 'ag_%s_step_host' % prefix)
    for k in range(2):
        a = _actions(k)
        ref = getattr(with_info, prefix + '_step_host')(a)
        obs, rew, done, _ = _outputs(obs_dim)
        assert fn(without.h, _p(a), _p(obs), _p(rew), _p(done), None) == 0, emu_lib.ag_last_error().decode()
        for x, y in zip((obs, rew, done), ref):
            np.testing.assert_array_equal(x, y)
    with_info.close(), without.close()
