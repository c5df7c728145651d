"""The stochastic policy sampled on the device, the parts that need no GPU: the numpy eps the GPU tests compare
with, the C ABI of the policy entry points, the registers of the policy step kernel, the CLI switch and the
tracker's pass plan."""
import ctypes
import os
import re
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from tests import noise_oracle as N
from tests import policy_oracle as PO
from tracktolearn_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NEW_SYMBOLS = ('ttl_env_step', 'ttl_policy_eps')


def test_policy_eps_is_independent_of_the_noise_under_one_seed():
    g = np.arange(20000, dtype=np.int64)
    L = (g % 37) + 1
    eps = PO.policy_eps(7, g, L)
    z = N.philox_normals(7, g, L)
    assert eps.dtype == np.float32 and eps.shape == (20000, 3)
    # counter words 3..5 are other draws than the noise's 0..2
    for a in range(3):
        for b in range(3):
            r = np.corrcoef(eps[:, a], z[:, b])[0, 1]
            assert abs(r) < 5 / np.sqrt(g.size), (a, b, r)
    # the fp32 rounding of the same Box-Muller transform
    np.testing.assert_array_equal(eps, PO.policy_normals(7, g, L).astype(np.float32))
    # a function of (seed, g, L) only, not of the position in the batch
    np.testing.assert_array_equal(PO.policy_eps(7, g[100:200], L[100:200]), eps[100:200])
    assert not np.array_equal(PO.policy_eps(8, g, L), eps)
    assert not np.array_equal(PO.policy_eps(7, g, L + 1), eps)
    assert not np.array_equal(PO.policy_eps(7, g + 2 ** 32, L), eps)


def test_policy_actions_at_prob_zero_are_tanh_mu():
    rs = np.random.RandomState(0)
    pre = rs.normal(size=(100, 6)).astype(np.float32)
    eps = rs.normal(size=(100, 3)).astype(np.float32)
    np.testing.assert_array_equal(PO.policy_actions(pre, eps, 0.0), np.tanh(pre[:, :3]))
    assert not np.array_equal(PO.policy_actions(pre, eps, 1.0), np.tanh(pre[:, :3]))


def test_policy_entry_points_are_exported_and_bound_in_abi_v5():
    build.build()
    lib = _lib.load()
    for name in NEW_SYMBOLS:
        assert hasattr(lib, name) and name in _lib.SIGNATURES, name
    header = open(os.path.join(ROOT, 'include', 'ttl_b200.h')).read()
    for name in NEW_SYMBOLS:
        assert re.search(r'\b%s\(' % name, header), name
    assert lib.ttl_abi_version() == _lib.ABI_VERSION


def test_policy_struct_layout_matches_header():
    src = r'''
#include "ttl_b200.h"
#include <stdio.h>
#include <stddef.h>
int main(void) {
  printf("%zu %zu %zu %zu\n", sizeof(ttl_policy), offsetof(ttl_policy, seed), offsetof(ttl_policy, row_base),
         offsetof(ttl_policy, prob));
  return 0;
}'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, 't.c')
        open(c, 'w').write(src)
        exe = os.path.join(d, 't')
        subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), c, '-o', exe])
        got = [int(x) for x in subprocess.check_output([exe]).split()]
    assert got == [ctypes.sizeof(_lib.Policy), _lib.Policy.seed.offset, _lib.Policy.row_base.offset,
                   _lib.Policy.prob.offset]


def test_policy_step_kernel_fits_six_ctas_per_sm_without_extra_stack():
    """Both builds of propagate_policy_kernel (with and without device noise) keep to the 80 registers of
    6 CTAs per SM, and their stack frame is no larger than the plain propagate_stop_kernel's (its 40-byte
    local array): no spills."""
    tool = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(tool):
        pytest.skip('cuobjdump not available')
    build.build()
    out = subprocess.run([tool, '-res-usage', _lib.LIB_PATH], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                         check=True).stdout.decode()

    def usage(kernel):
        return {b: (int(reg), int(stack)) for b, reg, stack in re.findall(
            r'Function \S*%sILb([01])E\S*:\s*\n\s*REG:(\d+) STACK:(\d+)' % kernel, out)}
    plain, policy = usage('propagate_stop_kernel'), usage('propagate_policy_kernel')
    assert set(policy) == {'0', '1'}, policy
    for b, (reg, stack) in policy.items():
        assert reg <= 80 and stack <= plain['0'][1], (b, policy, plain)


def _track_cli(args):
    return subprocess.run([sys.executable, os.path.join(ROOT, 'scripts', 'ttl_track.py')] + args,
                          stdout=subprocess.PIPE, stderr=subprocess.STDOUT)


def test_ttl_track_lists_policy_prob_and_rejects_a_negative_value(tmp_path):
    out = _track_cli(['--help'])
    assert out.returncode == 0 and '--policy_prob' in out.stdout.decode()
    files = [str(tmp_path / n) for n in ('fodf.nii.gz', 'seed.nii.gz', 'mask.nii.gz')]
    for f in files:
        open(f, 'wb').close()
    bad = _track_cli(files + [str(tmp_path / 'out.trk'), '--policy_prob', '-0.5'])
    assert bad.returncode == 2 and '--policy_prob' in bad.stdout.decode(), bad.stdout.decode()


class _Env(object):
    def __init__(self, n):
        self.seeds = np.zeros((n, 3))
        self.max_nb_steps = 100


def test_tracker_streams_a_seeded_stochastic_policy():
    from tracktolearn_b200.tracking.tracker import Tracker
    env = _Env(2500)
    batch = [(0, 1000, None), (1000, 2000, None), (2000, 2500, None)]
    assert list(Tracker(None, 1000, prob=0.0)._passes(env)) == [(0, 2500, 1000)]
    assert list(Tracker(None, 1000, prob=1.0)._passes(env)) == batch                  # torch.randn: batches
    assert list(Tracker(None, 1000, prob=1.0, policy_seed=3)._passes(env)) == [(0, 2500, 1000)]
    assert list(Tracker(None, 1000, prob=1.0, policy_seed=3, streaming=False)._passes(env)) == batch
