"""Out-of-bounds self-check (compute-sanitizer is closed on the GPU pool, profiles/r2_sanitizer_refused.txt):
every env buffer and the actor's workspace are carved out of larger allocations with 4 KB of 0xA5 on
either side; after whole episodes in every mode, at awkward sizes, no guard byte may have changed."""
import numpy as np
import pytest
import torch

from tracktolearn_b200 import synthetic

pytestmark = pytest.mark.gpu


@pytest.fixture
def guarded():
    from tracktolearn_b200.algorithms.shared.offpolicy import MaxEntropyActor
    from tracktolearn_b200.environments.tracking_env import _BatchBuffers
    old = (_BatchBuffers.GUARD, MaxEntropyActor.GUARD)
    _BatchBuffers.GUARD = MaxEntropyActor.GUARD = True
    yield
    _BatchBuffers.GUARD, MaxEntropyActor.GUARD = old


@pytest.mark.parametrize('n_seeds,slots', [(900, 256), (333, 31), (65, 64), (1, 1), (700, 33)])
def test_no_kernel_writes_outside_its_buffers(guarded, n_seeds, slots):
    from tests.test_tracker_gpu import _setup
    from tracktolearn_b200.algorithms.sac_auto import SACAuto
    env, alg32, sub, seeds, sd = _setup(n_seeds=n_seeds, precision='fp32')
    n = len(seeds)
    # reference protocol (fp32 rows + 16-bit copy, state of stopped rows), host actions
    st = env.reset(0, n)
    alg32.validation_episode(st, env, 0.0)
    assert env._batch.check_guards() == 0 and alg32.agent.actor.check_guards() == 0
    ref_lengths = env.lengths.copy()
    for prec in ('fp16', 'tf32', 'bf16'):
        alg = SACAuto(615, 3, '128-128-128', n_actors=slots, device=torch.device('cuda:0'), precision=prec)
        alg.agent.actor.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
        for fp32_state in (True, False):
            env._batch = None            # exact-size buffers: the guards border what the kernels may touch
            st = env.reset_streaming(0, n, slots, fp32_state=fp32_state, operand=prec)
            assert env._batch.GUARD and len(env._batch._guarded) > 15
            alg.validation_episode(st, env, 0.0)
            env.get_streamlines()
            assert env._batch.check_guards() == 0, (prec, fp32_state)
            assert alg.agent.actor.check_guards() == 0, (prec, fp32_state)
            if n >= 50:
                assert (env.lengths == ref_lengths).mean() > 0.85
