"""bench.py --dump-outputs: the state it writes is the API's state tensor whatever layout the actor's operand
rows use, so dumps of builds that lay those rows out differently still compare column for column."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_dumped_state_is_in_the_state_column_order():
    """Right after a streaming reset, the operand-only fp16 rows (channel-padded layout 1) come back in the
    same columns as the fp32 state rows of the reference layout, to fp16 rounding."""
    import bench
    from tests.test_tracker_gpu import _setup
    env, _, _, seeds, _ = _setup(precision='fp16')
    n, slots = len(seeds), 256
    dumps = {}
    for fp32_state in (True, False):
        env._batch = None
        env.reset_streaming(0, n, slots, fp32_state=fp32_state, operand='fp16')
        assert env.bf16_layout[0] == (0 if fp32_state else 1)
        dumps[fp32_state] = bench.capture_outputs(env, env.n_alive())
    ref, got = dumps[True], dumps[False]
    assert got['state'].shape == (slots, 615) and got['state_rows'].shape == (slots,)
    for k in ('lengths', 'flags', 'points', 'points_rows', 'alive_rows', 'state_rows'):
        np.testing.assert_array_equal(got[k], ref[k], err_msg=k)
    np.testing.assert_allclose(got['state'], ref['state'], rtol=2.0 ** -11, atol=1e-7)
    assert np.abs(ref['state']).max() > 0
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
