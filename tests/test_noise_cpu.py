"""Device-drawn tracking noise, the parts that need no GPU: the numpy Philox4x32-10 the GPU tests compare
with, the C ABI of the noise entry points, the registers of the RNG step kernel, the CLI switch and the env's argument checks."""
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
from tracktolearn_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# Random123's known-answer vectors for philox4x32_10 (kat_vectors): counter, key -> output
PHILOX_KAT = [
    ((0x00000000, 0x00000000, 0x00000000, 0x00000000), (0x00000000, 0x00000000),
     (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff, 0xffffffff, 0xffffffff, 0xffffffff), (0xffffffff, 0xffffffff),
     (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]


def test_numpy_philox_known_answers():
    for ctr, key, want in PHILOX_KAT:
        got = N.philox4x32_10(np.asarray(ctr), np.asarray(key))
        assert [int(v) for v in got] == list(want), [hex(int(v)) for v in got]
    # vectorised over a batch gives the same words
    ctr = np.asarray([c for c, _, _ in PHILOX_KAT])
    got = N.philox4x32_10(ctr[:2], np.asarray(PHILOX_KAT[0][1]))
    assert [int(v) for v in got[0]] == list(PHILOX_KAT[0][2])


def test_uniforms_stay_inside_the_open_interval():
    w = np.asarray([[0, 0, 0, 0], [0xffffffff] * 4, [0xfff, 0, 0x1000, 0]], dtype=np.uint32)
    u1, u2 = N.philox_uniforms(w)
    assert (u1 > 0).all() and (u1 < 1).all() and (u2 > 0).all() and (u2 < 1).all()
    assert u1[0] == 2.0 ** -53 and u1[1] == 1 - 2.0 ** -53
    assert u1[2] == u1[0]                   # the 12 low bits are dropped
    # the largest |z| the transform can produce
    z = np.sqrt(-2 * np.log(u1[0]))
    assert 8.57 < z < 8.58


def test_philox_normals_shape_and_dependence():
    g = np.arange(1000, dtype=np.int64)
    z = N.philox_normals(3, g, 5)
    assert z.shape == (1000, 3) and np.isfinite(z).all()
    np.testing.assert_array_equal(N.philox_normals(3, g[10:20], 5), z[10:20])   # a function of g, not position
    assert not np.array_equal(N.philox_normals(3, g, 6), z)
    assert not np.array_equal(N.philox_normals(4, g, 5), z)
    big = N.philox_normals(3, np.asarray([2 ** 40 + 7]), 5)                       # hi32(g) is part of the counter
    assert not np.array_equal(big, N.philox_normals(3, np.asarray([7]), 5))


def test_noise_entry_points_are_exported_and_bound_in_abi_v5():
    build.build()
    lib = _lib.load()
    for name in ('ttl_env_step', 'ttl_noise_normals'):
        assert hasattr(lib, name) and name in _lib.SIGNATURES, name
    assert lib.ttl_abi_version() == _lib.ABI_VERSION == 5


def test_noise_struct_layout_matches_header():
    src = r'''
#include "ttl_b200.h"
#include <stdio.h>
#include <stddef.h>
int main(void) {
  printf("%zu %zu %zu %zu\n", sizeof(ttl_noise), offsetof(ttl_noise, sigma), offsetof(ttl_noise, seed),
         offsetof(ttl_noise, row_base));
  return 0;
}'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, 't.c')
        open(c, 'w').write(src)
        exe = os.path.join(d, 't')
        subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), c, '-o', exe])
        got = [int(x) for x in subprocess.check_output([exe]).split()]
    assert got == [ctypes.sizeof(_lib.Noise), _lib.Noise.sigma.offset, _lib.Noise.seed.offset,
                   _lib.Noise.row_base.offset]


def test_rng_step_kernel_adds_no_stack_at_six_ctas_per_sm():
    """The RNG instantiation of propagate_stop_kernel, built for 6 CTAs per SM, fits the 80 registers
    that occupancy leaves without spilling: its stack frame is the plain instantiation's (a 40-byte local
    array both have), no larger."""
    tool = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(tool):
        pytest.skip('cuobjdump not available')
    build.build()
    out = subprocess.run([tool, '-res-usage', _lib.LIB_PATH], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                         check=True).stdout.decode()
    found = {b: (int(reg), int(stack)) for b, reg, stack in re.findall(
        r'Function \S*propagate_stop_kernelILb([01])E\S*:\s*\n\s*REG:(\d+) STACK:(\d+)', out)}
    assert set(found) == {'0', '1'}, found
    reg, stack = found['1']
    assert reg <= 80 and stack == found['0'][1], found


def test_ttl_track_help_lists_noise_rng():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'scripts', 'ttl_track.py'), '--help'],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, check=True).stdout.decode()
    assert '--noise_rng' in out and 'device' in out


def test_device_noise_needs_a_seed():
    from tracktolearn_b200.environments import NoisyTrackingEnvironment
    dto = {'noise': 0.1, 'noise_rng': 'device', 'fa_map': None}
    with pytest.raises(ValueError, match='noise_seed'):
        NoisyTrackingEnvironment(None, 'testing', dto)
    with pytest.raises(ValueError, match='noise_rng'):
        NoisyTrackingEnvironment(None, 'testing', dict(dto, noise_rng='gpu', noise_seed=1))
    with pytest.raises(ValueError, match='noise_seed'):
        NoisyTrackingEnvironment(None, 'testing', dict(dto, noise_seed=-1))
