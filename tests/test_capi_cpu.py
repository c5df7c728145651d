"""The C-ABI library loads without a GPU and exports every symbol include/ttl_b200.h declares;
the ctypes structures have the C layout."""
import ctypes
import os
import re
import subprocess
import tempfile

import pytest

from tracktolearn_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, 'include', 'ttl_b200.h')


def test_library_builds_and_exports_the_abi_v4_symbols():
    build.build()
    lib = _lib.load()
    text = open(HEADER).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    declared = set(re.findall(r'\b(ttl_[a-z0-9_]+)\s*\(', text))
    assert len(declared) >= 15
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    assert lib.ttl_abi_version() == _lib.ABI_VERSION == 4
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
            _lib.Batch.sg_stops.offset, _lib.Batch.operand_fmt.offset, _lib.Batch.order.offset]
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
