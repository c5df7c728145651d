#!/usr/bin/env python
"""ttl_track on N GPUs of one box writes the same tractogram as on one GPU.

    python benchmarks/multi_gpu_cli_check.py [N [ttl_track options...]]   # needs N visible GPUs (default 2)

e.g. ``2 --noise 0.1 --noise_rng device`` checks noisy tracking with device-drawn noise.

Builds a small synthetic subject on disk, runs the CLI in this process (1 GPU), runs it again under
``torch.distributed.run --nproc-per-node N`` (seeds sharded, NCCL gather to rank 0) and compares the
two files byte for byte after the header."""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    n = int(sys.argv[1]) if len(sys.argv) > 1 else 2
    from tracktolearn_b200 import synthetic
    from tracktolearn_b200.io import nifti
    from tracktolearn_b200.io.streamlines import read_tck, read_trk
    from tracktolearn_b200.runners.ttl_track import main as cli
    tmp = tempfile.mkdtemp(prefix='ttl_mgpu_')
    shape = (40, 44, 36)
    sub = synthetic.make_subject(shape, seed=5)
    affine = np.diag([1.25, 1.25, 1.25, 1.0])
    affine[:3, 3] = [-10.0, 4.0, 2.5]
    p = lambda f: os.path.join(tmp, f)  # noqa: E731
    nifti.save(p('fodf.nii.gz'), sub['sh'].numpy(), affine)
    nifti.save(p('mask.nii.gz'), sub['mask'].numpy(), affine)
    nifti.save(p('seed.nii.gz'), synthetic.ellipsoid_mask(shape, frac=0.3).numpy().astype(np.uint8), affine)
    agent = synthetic.write_agent_dir(p('agent'), kind='tracking', hidden_dims='256-256-256')
    out = {}
    for ext, reader in (('trk', read_trk), ('tck', read_tck)):
        common = [p('fodf.nii.gz'), p('seed.nii.gz'), p('mask.nii.gz')]
        opts = ['--agent', agent, '--hyperparameters', os.path.join(agent, 'hyperparameters.json'),
                '--n_actor', '3000', '--npv', '3', '--min_length', '5', '--max_length', '80', '--save_seeds',
                '--compress', '0.05', '-f'] + sys.argv[2:]
        one = p('one.' + ext)
        cli(common + [one] + opts)
        many = p('many.' + ext)
        cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(n),
               '--master-addr', '127.0.0.1', '--master-port', '29561', os.path.join(ROOT, 'scripts', 'ttl_track.py')]
        subprocess.check_call(cmd + common + [many] + opts, stdout=subprocess.DEVNULL)
        d1, o1, _ = reader(one)
        d2, o2, _ = reader(many)
        same = bool(np.array_equal(o1, o2) and np.array_equal(d1, d2))
        out[ext] = {'streamlines': int(len(o1) - 1), 'points': int(len(d1)), 'identical': same}
        assert same, ext
    print(json.dumps({'gpus': n, 'options': sys.argv[2:], 'result': out}))


if __name__ == '__main__':
    main()
