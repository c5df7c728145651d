"""The C-ABI library loads without a GPU and exports every symbol include/ttl_b200.h declares;
the ctypes structures have the C layout."""
import ctypes
import json
import os
import re
import subprocess
import sys
import tempfile

import pytest

from tracktolearn_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, 'include', 'ttl_b200.h')


def test_library_builds_and_exports_the_abi_v5_symbols():
    build.build()
    lib = _lib.load()
    text = open(HEADER).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    declared = set(re.findall(r'\b(ttl_[a-z0-9_]+)\s*\(', text))
    assert len(declared) >= 15
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert lib.ttl_abi_version() == _lib.ABI_VERSION == 5
    assert lib.ttl_launch_count() >= 0


def test_ctypes_struct_layout_matches_header():
    src = r'''
#include "ttl_b200.h"
#include <stdio.h>
#include <stddef.h>
int main(void) {
  printf("%zu %zu %zu %zu %zu %zu %zu %zu\n", sizeof(ttl_volume), sizeof(ttl_params), sizeof(ttl_batch),
         sizeof(ttl_actor_weights), sizeof(ttl_oracle_weights), offsetof(ttl_batch, alive),
         offsetof(ttl_batch, state), offsetof(ttl_params, theta_rad));
  printf("%zu %zu %zu\n", offsetof(ttl_batch, sg_stops), offsetof(ttl_batch, operand_fmt), offsetof(ttl_batch, order));
  printf("%zu %zu %zu %zu %zu %zu\n", sizeof(ttl_step_action), offsetof(ttl_step_action, head_partial),
         offsetof(ttl_step_action, head_bias), offsetof(ttl_step_action, lda), offsetof(ttl_step_action, n_tiles),
         offsetof(ttl_step_action, tiles_per_256));
  return 0;
}'''
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, 't.c')
        open(c, 'w').write(src)
        exe = os.path.join(d, 't')
        subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), c, '-o', exe])
        got = [int(x) for x in subprocess.check_output([exe]).split()]
    want = [ctypes.sizeof(_lib.Volume), ctypes.sizeof(_lib.Params), ctypes.sizeof(_lib.Batch),
            ctypes.sizeof(_lib.ActorWeights), ctypes.sizeof(_lib.OracleWeights),
            _lib.Batch.alive.offset, _lib.Batch.state.offset, _lib.Params.theta_rad.offset,
            _lib.Batch.sg_stops.offset, _lib.Batch.operand_fmt.offset, _lib.Batch.order.offset,
            ctypes.sizeof(_lib.StepAction), _lib.StepAction.head_partial.offset, _lib.StepAction.head_bias.offset,
            _lib.StepAction.lda.offset, _lib.StepAction.n_tiles.offset, _lib.StepAction.tiles_per_256.offset]
    assert got == want


def test_product_refuses_cpu_device():
    import numpy as np
    import pytest
    import torch
    from tracktolearn_b200.algorithms.shared.offpolicy import SACActorCritic
    with pytest.raises(_lib.TTLError):
        SACActorCritic(615, 3, '64-64-64', torch.device('cpu'))


def test_tensor_core_kernels_keep_their_registers():
    """A tcgen05 epilogue whose TMEM read buffers fall out of registers into local memory still gives
    right answers but runs at half speed (measured: 61 -> 112 us per layer).  ptxas reports it as a
    stack frame, so pin STACK:0 for the dense kernels in the built library."""
    import re
    import shutil
    import subprocess
    tool = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(tool):
        pytest.skip('cuobjdump not available')
    out = subprocess.run([tool, '-res-usage', _lib.LIB_PATH], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                         check=True).stdout.decode()
    found = re.findall(r'Function (\S*mlp_pair_kernel\S*):\s*\n\s*REG:(\d+) STACK:(\d+)', out)
    assert len(found) == 6, found          # {bf16, fp16, tf32} x {plain, fused head}
    for name, reg, stack in found:
        assert int(stack) == 0, (name, reg, stack)


_STEP_ARGS_PROBE = r'''
import ctypes, json, sys
sys.path.insert(0, sys.argv[1])
from tracktolearn_b200 import _lib
lib = _lib.load()
fake = iter(range(1 << 20, 1 << 30, 1 << 16))          # distinct 256-byte aligned addresses, never dereferenced
vol = _lib.Volume(sh=next(fake), X=8, Y=8, Z=8, C=45, CP=48, mask_coef=next(fake), MX=8, MY=8, MZ=8)
prm = _lib.Params(step_vox=0.5, mask_threshold=0.5, theta_rad=0.5, max_nb_steps=100, n_dirs=100, dir_f64=1)
b = _lib.Batch(n=1000, n_slots=1000, capacity=1000, max_pts=101, ld_state=616, state_size=615, ld_bf16=640,
               max_groups=33, grp_stops=next(fake), sg_stops=next(fake), step_tip=next(fake), operand_fmt=0)
for f in ('points', 'flags', 'lengths', 'npts', 'dones', 'ctrl', 'stop', 'dest', 'step_flags', 'reward'):
    setattr(b, f, next(fake))
for f in ('alive', 'state', 'state_bf16', 'rank_rec'):
    getattr(b, f)[0], getattr(b, f)[1] = next(fake), next(fake)
actions = dict(actions=next(fake), lda=3)
head = dict(head_partial=next(fake), head_bias=next(fake), n_tiles=4, tiles_per_256=1)
noise, nz, pol = ctypes.c_void_p(next(fake)), _lib.Noise(sigma=0.1, seed=1), _lib.Policy(seed=1, prob=1.0)


def step(act, noise=None, nz=None, pol=None, defer=0):
    return lib.ttl_env_step(vol, prm, b, 0, None if act is None else _lib.StepAction(**act), noise,
                            None if nz is None else ctypes.byref(nz), None if pol is None else ctypes.byref(pol),
                            defer, 64, None)


codes = {
    'no action struct': step(None),
    'both action sources': step(dict(actions, **head)),
    'neither action source': step({}),
    'noise array with device noise': step(actions, noise=noise, nz=nz),
    'policy with an action buffer': step(actions, pol=pol),
    'fused head with a noise array': step(head, noise=noise),
    'fused head deferred': step(head, defer=1),
    'fused head with policy deferred': step(head, pol=pol, defer=1),
    'defer other than 0 or 1': step(actions, defer=2),
}
prm.dir_f64 = 0
codes['device noise without float64 directions'] = step(head, nz=nz)
prm.dir_f64 = 1
codes['accepted'] = [step(actions, nz=nz, defer=1), step(head, nz=nz, pol=pol)]   # reach the first CUDA call
print(json.dumps(codes))
'''


def test_env_step_rejects_every_combination_it_does_not_serve():
    """ttl_env_step serves the action buffer (host noise or device noise, deferred for the oracle or not) and
    the fused head (device noise, with or without the sampled policy, never deferred).  Every other
    combination is refused before any CUDA call, with host structs that pass every other check and
    n_upper > 0.  No device is made visible to the probe: a combination that got through would fail its
    first CUDA call instead of launching on the fake pointers."""
    build.build()
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')
    out = subprocess.run([sys.executable, '-c', _STEP_ARGS_PROBE, ROOT], env=env, stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT)
    assert out.returncode == 0, out.stdout.decode()
    codes = json.loads(out.stdout.decode().strip().splitlines()[-1])
    assert all(c > 0 for c in codes.pop('accepted')), codes      # a CUDA error: the structs pass every check
    assert codes.pop('device noise without float64 directions') == -2
    assert len(codes) == 9 and all(c == -1 for c in codes.values()), codes
