#!/usr/bin/env python
"""bench.py -- streamline-steps/sec of the batched tracking step on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--precision fp16|tf32|bf16]
                    [--dump-outputs DIR]

Workload (BASELINE.json configs[1], the configuration the metric is quoted on): whole-brain synthetic
145x174x145 1.25 mm order-8 descoteaux07 fODF, npv 20 on the mask shell (873 000 seeds per GPU),
n_actor 50 000, NoisyTrackingEnvironment with noise 0 (what ttl_track.py always runs), SAC actor
615-1024-1024-1024-6 with a synthetic "tracking-like" checkpoint.  One bench STEP = one pass of the hot
path over the batch of n_actor alive streamlines: actor forward (ONE persistent tcgen05 launch for the
three hidden layers with the 6-wide head fused into the last) + env step (propagate / stopping criteria
with the head's tanh finish, then the state gather with ordered compaction, slot refill and control-block
update) -- 3 kernel launches, no host involvement.

What the JSON line carries (DESIGN.md section 6 says how every field is produced):
  value        device-resident steady-state throughput of the headline tier (fp16 operands: within the
               1e-3 tolerance at the full 16-bit tensor rate), timed on a rested chip: 384 burn-in steps,
               2 s of idle, W warm-up steps, K timed steps; `tiers` holds the same measurement for tf32
               (1e-3, fp32 range, half rate) and bf16 (4e-3, outside the tolerance)
  sustained    the headline tier again after ~125 ms of continuous load (what sw_power_cap leaves)
  e2e          Tracker over 800 000 seeds per GPU from pinned host seeds to host-resident packed
               streamlines; with N > 1 the seeds are one list, shuffled once and sharded, and the timed
               region ends with the NCCL gather of every rank's streamlines on rank 0
  sharded      BASELINE.json configs[2]: 290^3 0.5 mm volume, exactly 1 000 000 seeds sharded over the N
               GPUs (strong scaling), tracked end to end and gathered on rank 0
  roofline     the tcgen05 launch against the burst peak of its operand type
  cpu_baseline the CPU restatement of the reference path on the host cores, same 50 000-row batch
`--impl reference` times that CPU restatement (oracle/ttl_oracle.py + a torch-CPU fp32 actor) alone, under
the better of OMP_NUM_THREADS in {1, cores}.

`--dump-outputs DIR` writes, on rank 0, what the headline tier's timed steps left a caller after the last
of them, as DIR/<name>.npy (float32 / float64, integers stored exactly as float64, under 64 MB in all):
  lengths, flags        [N]                 every row (seed) of the batch
  points, points_rows   [4096, max_pts, 3]  the streamline buffer of a fixed, seeded sample of rows
  alive_rows            [n_alive]           the rows still tracked, ascending
  state, state_rows     [8192, 615]         the actor's next input for a fixed, seeded sample of those rows,
                                            in the state's column order, at the operand precision
The inputs (volume, seeds, actor) are seeded, so two builds run with the same arguments can be compared
array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SHAPE = (145, 174, 145)
VOXEL_MM = 1.25
NPV = 20
N_ACTOR = 50000
TRAINED_VOXEL = 0.9987237            # models/hyperparameters.json:49
TRAINED_STEP = 0.75
STEP_MM = VOXEL_MM / TRAINED_VOXEL * TRAINED_STEP   # runners/ttl_track.py:126-141
MAX_LENGTH_MM = 300.0                # ttl_track.py --max_length default
THETA = 30.0
HIDDEN = '1024-1024-1024'
STATE_SIZE = 615
ACTOR_FLOP_PER_ROW = 2 * (615 * 1024 + 2 * 1024 * 1024 + 1024 * 6)      # SURVEY 8(d): 5 466 112
DENSE_FLOP_PER_ROW = 2 * (615 * 1024 + 2 * 1024 * 1024)                 # the three tcgen05 layers
WORKLOAD = 'whole-brain synthetic 145x174x145 1.25mm order-8 fODF, npv=20, n_actor=50000'
BURN_IN = 384
TF32_NOMINAL_TFLOPS = 1100.0
REST_S = 2.0            # idle between the burn-in and the warm-up steps of every leg (see run_tier)
SUSTAIN_STEPS = 400     # continuous load before the `sustained` measurement of every leg (~125 ms)
E2E_SEEDS = 16 * N_ACTOR
SHARDED_SHAPE = (290, 290, 290)
SHARDED_VOXEL_MM = 0.5
SHARDED_SEEDS = 1000000
TIERS = ('fp16', 'tf32', 'bf16')
TIER_NOTE = {
    'fp16': 'fp16 operands (11 significant bits), fp32 accumulate: actor outputs within 1e-3 of the fp32 reference',
    'tf32': 'tf32 operands (11 significant bits, fp32 range), fp32 accumulate: within 1e-3, half the tensor rate',
    'bf16': 'bf16 operands (8 significant bits): ~4e-3 of the output scale, OUTSIDE the 1e-3 tolerance',
}
NCU_SUMMARY = os.path.join(ROOT, 'profiles', 'r2_final_step_ncu_summary.json')
DUMP_POINTS_ROWS = 4096
DUMP_STATE_ROWS = 8192
DUMP_MAX_BYTES = 64 << 20


def workload_config(shape=SHAPE, voxel_mm=VOXEL_MM):
    """The `config` object both arms print: what is computed, nothing about how or where."""
    step_mm = voxel_mm / TRAINED_VOXEL * TRAINED_STEP
    return {'workload': WORKLOAD, 'volume': list(shape), 'voxel_mm': voxel_mm, 'npv': NPV, 'n_actor': N_ACTOR,
            'step_mm': step_mm, 'max_nb_steps': int(MAX_LENGTH_MM / step_mm), 'theta': THETA,
            'actor': '615-' + HIDDEN + '-6 (synthetic, tracking-like)',
            'env': 'NoisyTrackingEnvironment noise=0 (float64 directions)',
            'rows_per_step': N_ACTOR}


def ncu_traffic():
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the step's kernels from
    the committed `ncu --set full` capture of this same command (profiles/README.md); {} when the
    summary file is absent."""
    if not os.path.exists(NCU_SUMMARY):
        return {}

    def mbytes(txt):
        v, unit = txt.split()[:2]
        return float(v) * {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}[unit]
    per = {}
    with open(NCU_SUMMARY) as f:
        for e in json.load(f):
            name = e['kernel'].split('<')[0].split('(')[0]
            per.setdefault(name, []).append(mbytes(e['dram__bytes_read.sum']) + mbytes(e['dram__bytes_write.sum']))
    return {k: sum(v) / len(v) for k, v in per.items()}


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {'hbm_gbs': p['hbm_gbs'], 'bf16_tflops': p['bf16_tflops'],
                'bf16_tflops_sustained': p.get('bf16_tflops_sustained', p['bf16_tflops']),
                'source': 'measured (MEASURED_PEAKS.json)'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0,
            'source': 'fallback (B200_PROFILING.md)'}


def measure_tf32_peak(dev):
    """cuBLAS TF32 8192^3, best of 10 (the way MEASURED_PEAKS.json's bf16 burst figure was taken): the
    denominator of the tf32 tier's roofline.  ~25 ms."""
    import torch
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        a = torch.randn((8192, 8192), device=dev)
        b = torch.randn((8192, 8192), device=dev)
        best = float('inf')
        for i in range(13):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            torch.cuda.synchronize(dev)
            if i >= 3:
                best = min(best, e0.elapsed_time(e1))
        return 2.0 * 8192 ** 3 / (best * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q,
                 '--format=csv,noheader,nounits', '-lms', '10'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.monotonic(), line.strip()))

    def wait_first(self, timeout_s):
        """Block until nvidia-smi has produced its first sample (it starts slowly)."""
        t0 = time.monotonic()
        while self.proc is not None and not self.rows and time.monotonic() - t0 < timeout_s:
            time.sleep(0.01)

    def mark_begin(self):
        self.t_begin = time.monotonic()

    def mark_end(self):
        self.t_end = time.monotonic()

    def median_between(self, t0, t1):
        """Median SM clock of the samples read in [t0, t1 + 40 ms] (None when there is none)."""
        sm = []
        for (t, r) in list(self.rows):
            if t0 <= t <= t1 + 0.04:
                f = [x.strip() for x in r.split(',')]
                try:
                    sm.append(float(f[1]))
                except (ValueError, IndexError):
                    pass
        return float(np.median(sm)) if sm else None

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        t0, t1 = getattr(self, 't_begin', 0.0), getattr(self, 't_end', float('inf'))
        # a sample is read ~one period after it was taken: accept rows up to 40 ms past the end mark;
        # a timed region shorter than the sampling period falls back to the nearest samples around it
        rows = [r for (t, r) in self.rows if t0 <= t <= t1 + 0.04]
        window = 'timed region'
        if len(rows) < 2:
            rows = [r for (t, r) in self.rows if t0 - 0.1 <= t <= t1 + 0.1]
            window = 'timed region +-100 ms (region shorter than the sampling period)'
        sm, smax, reasons = [], [], set()
        for r in rows:
            f = [x.strip() for x in r.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'),
                                 f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None,
                'sm_max_mhz': float(max(smax)) if smax else None,
                'reasons': sorted(reasons), 'samples': len(sm), 'window': window}



# ------------------------------------------------------------------------------------------
# CPU arm: the reference path restated (oracle) with a torch-CPU actor on the host cores
# ------------------------------------------------------------------------------------------
CPU_PHASES = ('actor_forward', 'format_state', 'mask_spline', 'curvature_length', 'bookkeeping')


def cpu_reference_run(sub_np, seeds, actor_sd, rows, steps, warmup):
    """`steps` act -> step -> harvest iterations over `rows`-streamline batches; returns
    (streamline-steps/s, torch threads, ms per step, seconds per phase)."""
    import torch
    from oracle import ttl_oracle as O
    threads = torch.get_num_threads()
    W = [(actor_sd['layers.%d.weight' % (2 * i)].float(), actor_sd['layers.%d.bias' % (2 * i)].float())
         for i in range(4)]
    phase = dict.fromkeys(CPU_PHASES, 0.0)
    timing = {'on': False}

    def timed(name, fn):
        def wrapper(*a, **k):
            t0 = time.perf_counter()
            out = fn(*a, **k)
            if timing['on']:
                phase[name] += time.perf_counter() - t0
            return out
        return wrapper

    def torch_actor(state):      # offpolicy.py:94-140 at probabilistic = 0
        with torch.no_grad():
            h = torch.from_numpy(state)
            for i, (w, b) in enumerate(W):
                h = torch.addmm(b, h, w.t())
                if i < 3:
                    h = torch.relu(h)
            return torch.tanh(h[:, :3]).numpy()
    torch_actor = timed('actor_forward', torch_actor)

    env = O.OracleEnv(sub_np['sh'], sub_np['mask'], seeds, VOXEL_MM, STEP_MM, theta=THETA,
                      max_length_mm=MAX_LENGTH_MM, noisy=True)
    # per-phase split (BASELINE.md section 3): wrap the env's own methods, the arithmetic is untouched
    env._format_state = timed('format_state', env._format_state)
    env.mask_criterion = timed('mask_spline', env.mask_criterion)
    env._is_stopping = timed('curvature_length', env._is_stopping)       # minus mask_spline, below
    state = env.reset(0, rows)
    total, t_total, it, start_pos = 0, 0.0, 0, rows
    per_step = []
    while it < warmup + steps:
        if len(env.continue_idx) == 0:
            end = min(start_pos + rows, len(seeds))
            if end <= start_pos:
                start_pos, end = 0, rows
            state = env.reset(start_pos, end)
            start_pos = end
        timing['on'] = it >= warmup
        t0 = time.perf_counter()
        n = len(env.continue_idx)
        action = torch_actor(state)
        env.step(action)
        state, _ = env.harvest()
        dt = time.perf_counter() - t0
        if it >= warmup:
            total += n
            t_total += dt
            per_step.append(dt)
        it += 1
    phase['curvature_length'] -= phase['mask_spline']
    phase['bookkeeping'] = t_total - sum(phase[k] for k in CPU_PHASES if k != 'bookkeeping')
    return total / t_total, threads, 1000.0 * t_total / max(1, len(per_step)), phase


def build_subject_numpy():
    from tracktolearn_b200 import synthetic
    sub = synthetic.make_subject(SHAPE, seed=1234, with_peaks=False)
    return {k: (v.numpy() if v is not None else None) for k, v in sub.items()}


def draw_seeds(seed_mask, rank):
    """npv = 20 seeds per shell voxel (873 000), the share of rank `rank`."""
    from tracktolearn_b200.environments.utils import random_seeds_from_mask
    rs = np.random.RandomState(1337 + rank)
    return random_seeds_from_mask(seed_mask, NPV, rs)


def sharded_seed_list(seed_mask, world, rank):
    """ONE seed list for the whole job -- npv = 20 per GPU over the mask shell (weak scaling: 873 000
    seeds per GPU) -- shuffled once with a common RNG (tracking/tracker.py:94) and sharded in contiguous
    slices (parallel.shard_seeds).  Every rank builds the same list and keeps its slice."""
    from tracktolearn_b200 import parallel
    seeds = np.concatenate([draw_seeds(seed_mask, r) for r in range(world)])
    np.random.RandomState(4242).shuffle(seeds)
    return parallel.shard_seeds(seeds, rank, world)


def cpu_worker(args):
    """One CPU measurement in a fresh process (OMP_NUM_THREADS is read when numpy / torch load)."""
    import torch
    d = args.cpu_worker
    sub = {'sh': np.load(os.path.join(d, 'sh.npy'), mmap_mode='r'), 'mask': np.load(os.path.join(d, 'mask.npy'))}
    seeds = np.load(os.path.join(d, 'seeds.npy'))
    sd = torch.load(os.path.join(d, 'actor.pt'))
    torch.set_num_threads(args.torch_threads)
    v, threads, ms, phase = cpu_reference_run(sub, seeds, sd, N_ACTOR, args.steps, args.warmup)
    sys.stdout.write(json.dumps({'value': v, 'threads': threads, 'ms_per_step': ms, 'phase_s': phase,
                                 'omp': os.environ.get('OMP_NUM_THREADS')}) + '\n')
    return 0


def cpu_reference_best(sub_np, seeds, actor_sd, steps, warmup, probe_steps=2):
    """The CPU arm under the better of OMP_NUM_THREADS in {1, cores}: torchrun exports
    OMP_NUM_THREADS=1, a bare launch leaves it unset, and the numpy / OpenBLAS / torch thread pools
    oversubscribe each other by 3x in the wrong setting -- so both are tried on a short probe, each in
    its own process, and the timed run uses the winner.  torch's intra-op pool always has all cores.
    Returns (result dict of the timed run, description of the choice)."""
    cores = os.cpu_count() or 1
    with tempfile.TemporaryDirectory(prefix='ttl_bench_cpu_') as d:
        import torch
        np.save(os.path.join(d, 'sh.npy'), np.ascontiguousarray(sub_np['sh']))
        np.save(os.path.join(d, 'mask.npy'), np.ascontiguousarray(sub_np['mask']))
        np.save(os.path.join(d, 'seeds.npy'), seeds)
        torch.save(actor_sd, os.path.join(d, 'actor.pt'))

        def run(omp, k, w):
            env = dict(os.environ)
            env['OMP_NUM_THREADS'] = str(omp)
            env.pop('MKL_NUM_THREADS', None)
            p = subprocess.run([sys.executable, os.path.abspath(__file__), '--cpu-worker', d, '--steps', str(k),
                                '--warmup', str(w), '--torch-threads', str(cores)],
                               stdout=subprocess.PIPE, stderr=subprocess.PIPE, env=env)
            if p.returncode != 0:
                raise RuntimeError('cpu worker failed: ' + p.stderr.decode()[-2000:])
            return json.loads(p.stdout.decode().strip().splitlines()[-1])
        settings = [1] if cores == 1 else [1, cores]
        probes = {omp: run(omp, probe_steps, 1)['value'] for omp in settings}
        best = max(probes, key=probes.get)
        res = run(best, steps, warmup)
    choice = {'OMP_NUM_THREADS': best, 'torch_threads': cores,
              'probe_streamline_steps_per_s': {str(k): v for k, v in probes.items()}}
    return res, choice


def main_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return 0
    from tracktolearn_b200 import synthetic
    sub = build_subject_numpy()
    seeds = sharded_seed_list(sub['seed_mask'], 1, 0)
    sd = synthetic.actor_state_dict(STATE_SIZE, HIDDEN, seed=1111, kind='tracking')
    res, choice = cpu_reference_best(sub, seeds, sd, args.steps, args.warmup)
    value = res['value']
    sample = ('%d act->step->harvest iterations (after %d warm-up) over the same %d-streamline batch of the same '
              'volume and seeds as the GPU arm (numpy/scipy env restatement + torch-CPU fp32 actor; scipy '
              'map_coordinates is single-threaded)' % (args.steps, args.warmup, N_ACTOR))
    line = {
        'impl': 'reference', 'metric': 'streamline-steps/sec', 'value': value, 'unit': 'streamline-steps/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': res['ms_per_step'],
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        'config': workload_config(),
        'cpu_baseline': {'value': value, 'unit': 'streamline-steps/s', 'cores': os.cpu_count() or 1, 'kind': 'port',
                         'sample': sample, 'threads': choice, 'phase_seconds': res['phase_s']},
        'e2e': {'value': value, 'unit': 'streamline-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    emit(line)
    return 0


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version
    banner on stdout from C): point fd 1 at stderr for the run and keep the real stdout for the line."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), 'w')
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + '\n')
    out.flush()


def make_env(shape, voxel_mm, dev):
    import torch
    from tracktolearn_b200 import synthetic
    from tracktolearn_b200.datasets.utils import MRIDataVolume
    from tracktolearn_b200.environments import NoisyTrackingEnvironment
    sub = synthetic.make_subject(shape, seed=1234, device=dev, with_peaks=False)
    affine = np.diag([voxel_mm] * 3 + [1.0])
    subject = (MRIDataVolume(sub['sh'], affine), MRIDataVolume(sub['mask'], affine),
               MRIDataVolume(sub['seed_mask'], affine), None, affine)
    dto = {'n_dirs': 100, 'theta': THETA, 'npv': 1, 'binary_stopping_threshold': 0.1,
           'step_size': voxel_mm / TRAINED_VOXEL * TRAINED_STEP, 'min_length': 10.0, 'max_length': MAX_LENGTH_MM,
           'oracle_checkpoint': None, 'oracle_stopping_criterion': False, 'scoring_data': None,
           'compute_reward': False, 'alignment_weighting': 0.0, 'oracle_bonus': 0.0,
           'rng': np.random.RandomState(1337), 'device': dev, 'target_sh_order': 8,
           'noise': 0.0, 'fa_map': None, 'state_of_stopped': False}
    env = NoisyTrackingEnvironment(subject, 'testing', dto)
    return env, sub


def state_columns(env):
    """Column of each state feature in the actor's operand rows: layout 1 pads every neighbourhood point's C
    coefficients to CP columns (include/ttl_b200.h, ttl_batch.bf16_layout)."""
    layout, C, CP, n_points = env.bf16_layout
    S = env._batch.state_size
    if layout == 0:
        return np.arange(S)
    return np.concatenate([p * CP + np.arange(C) for p in range(n_points)] + [n_points * CP + np.arange(S - n_points * C)])


def capture_outputs(env, n_alive):
    """Host copies of what the step path left a caller after its last step (see --dump-outputs)."""
    import torch
    bb = env._batch
    n = env._n
    rs = np.random.RandomState(2024)
    pts_rows = np.sort(rs.choice(n, min(n, DUMP_POINTS_ROWS), replace=False))
    alive = bb.alive[env._cur][:n_alive].long()
    alive_sorted, ranks = torch.sort(alive)
    pick = torch.from_numpy(np.sort(rs.choice(n_alive, min(n_alive, DUMP_STATE_ROWS), replace=False))).to(env.device)
    st = env.current_state()
    if st is None:        # operand-only rows: back to the state's column order
        st = env.current_state_bf16()[:, torch.from_numpy(state_columns(env)).to(env.device)]
    out = {'lengths': bb.lengths[:n].double(), 'flags': bb.flags[:n].double(),
           'points': bb.points[torch.from_numpy(pts_rows).to(env.device)].float(),
           'points_rows': torch.from_numpy(pts_rows).double(), 'alive_rows': alive_sorted.double(),
           'state': st[ranks[pick]].float(), 'state_rows': alive_sorted[pick].double()}
    return {k: v.cpu().numpy() for k, v in out.items()}


def write_outputs(d, outputs):
    total = sum(a.nbytes for a in outputs.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError('--dump-outputs: %d bytes exceeds the %d byte limit' % (total, DUMP_MAX_BYTES))
    os.makedirs(d, exist_ok=True)
    for name, a in outputs.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(d, name + '.npy'), a)


def roofline_of(prec, prof, rows, pk, tf32_peak, traffic):
    """The tcgen05 launch(es) of one step against the burst peak of the operand type.  The per-launch
    time comes from CUDA events bracketing every launch of the library (ttl_prof_enable) in a separate
    ~6 ms segment right after the timed region: a kernel timed in a window that short runs at burst
    clocks, so the burst figure is the denominator (the sustained one is printed beside it)."""
    names = ('mlp_fused_head_kernel', 'mlp_fused_kernel', 'dense_kernel', 'dense_head_kernel')
    dn = [prof.get(k, (0, 0.0)) for k in names]
    launches = sum(n for n, _ in dn)
    total_ms = sum(ms for _, ms in dn)
    if not launches:
        return None
    per_step = 1 if (prof.get('mlp_fused_head_kernel') or prof.get('mlp_fused_kernel')) else 3
    steps_prof = launches / float(per_step)
    achieved = DENSE_FLOP_PER_ROW * rows * steps_prof / (total_ms * 1e-3) / 1e12
    if prec == 'tf32':
        # MEASURED_PEAKS.json holds no TF32 figure.  Two measured candidates -- cuBLAS' TF32 GEMM timed in this
        # run, and half the measured 16-bit burst peak (kind::tf32 issues at half the kind::f16 rate) -- have
        # both come out BELOW what this kernel sustains on a rested chip (846 vs 760 and 823 TFLOP/s), so
        # neither bounds it; the denominator is the hardware's nominal dense TF32 rate (B200_PROFILING.md's
        # table, 1.1 PFLOP/s), and the two measured figures are printed beside it.
        peak = TF32_NOMINAL_TFLOPS
        src = ('nominal dense TF32 rate (B200_PROFILING.md table); measured for comparison: cuBLAS TF32 matmul '
               '8192^3 in this run, best of 10: %.1f; half the measured 16-bit burst peak: %.1f'
               % (tf32_peak, pk['bf16_tflops'] / 2.0))
    else:
        peak, src = pk['bf16_tflops'], pk['source'] + ', burst 16-bit figure (kernel timed alone in a ~6 ms window)'
    r = {'kernel': 'mlp_pair_kernel<%s> (tcgen05 cta_group::2, %d launch%s per step for the three hidden layers, '
                   '6-wide head fused into the last)' % (prec, per_step, '' if per_step == 1 else 'es'),
         'bound': 'tensor', 'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s', 'frac': achieved / peak,
         'traffic': traffic.get('mlp_pair_kernel'), 'traffic_source': os.path.relpath(NCU_SUMMARY, ROOT)
         if traffic else None,
         'avg_launch_us': 1000.0 * total_ms / launches, 'flop_per_launch': DENSE_FLOP_PER_ROW * rows / float(per_step),
         'peak_source': src}
    if prec != 'tf32':
        r['frac_of_sustained_peak'] = achieved / pk['bf16_tflops_sustained']
    else:
        r['achieved_over_cublas_tf32'] = achieved / tf32_peak if tf32_peak else None
    return r


def run_tier(env, actor_sd, prec, args, dev, lib, barrier, sampler=None, is_main=False):
    """Device-resident steady state of one precision tier: inputs already in HBM, K timed steps."""
    import torch
    from tracktolearn_b200 import _lib
    from tracktolearn_b200.algorithms.rl import StepRunner
    from tracktolearn_b200.algorithms.sac_auto import SACAuto
    alg = SACAuto(STATE_SIZE, 3, HIDDEN, n_actors=N_ACTOR, device=dev, precision=prec)
    alg.agent.actor.load_state_dict(actor_sd)
    actor = alg.agent.actor
    stream = torch.cuda.current_stream(dev)
    n_seeds = len(env.seeds)
    env.reset_streaming(0, n_seeds, N_ACTOR, fp32_state=not args.operand_only, operand=prec)
    runner = StepRunner(env, actor, 0.0, use_graph=args.graph)
    # burn-in (untimed, part of preparing the workload): with slot refill the alive set needs about
    # two mean lifetimes to reach its steady-state mix of streamline ages and positions; right after
    # reset every streamline still sits on the seed shell and the gather enjoys unrepresentative L2
    # locality.  Those 384 steps are ~120 ms of full load, and on this pool sw_power_cap can pull the SM
    # clock from 1965 to ~1600 MHz within ~100 ms of continuous load (all three kernels slow down alike:
    # scripts/gpu_ab_old.sh -- the same binary 155 M and 180 M in consecutive processes;
    # benchmarks/ramp_probe.py -- 305 us/step right after the burn-in, 264 us for every later burst).
    # The timed region therefore starts from a RESTED chip: burn-in, REST_S of idle, W warm-up steps, K
    # timed steps -- the regime MEASURED_PEAKS.json's burst figures (the roofline denominators) were taken
    # in.  What the same tier does under continuous load is reported beside it (`sustained`), and `e2e`
    # is a 270 ms continuous run by construction.
    for _ in range(BURN_IN):
        runner.step()
    env.n_alive()
    time.sleep(REST_S)
    for _ in range(args.warmup):
        runner.step()
    env.n_alive()
    steps_before = env.streamline_steps()
    launches_before = lib.ttl_launch_count()
    replays_before = runner.replays
    barrier()
    if sampler is not None:
        sampler.wait_first(2.0)
        if is_main:
            sampler.mark_begin()
    t_begin = time.monotonic()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        runner.step()
    ev1.record(stream)
    barrier()
    t_end = time.monotonic()
    if sampler is not None and is_main:
        sampler.mark_end()
    elapsed_ms = ev0.elapsed_time(ev1)
    # kernels launched one by one + kernels replayed from the captured step graphs
    gpu_launches = int(lib.ttl_launch_count() - launches_before) + \
        (runner.replays - replays_before) * runner.kernels_per_step
    env.n_alive()
    units = env.streamline_steps() - steps_before
    alive_end = int(env._batch.ctrl_host[env._cur])
    outputs = capture_outputs(env, alive_end) if args.dump_outputs and is_main else None
    # per-kernel device times (CUDA events on the launching stream), separate segment
    prof_steps = min(20, args.steps)
    lib.ttl_prof_enable(1)
    plain = StepRunner(env, actor, 0.0, use_graph=False)
    for _ in range(prof_steps):
        plain.step()
    torch.cuda.synchronize(dev)
    prof = _lib.prof_report()
    lib.ttl_prof_enable(0)
    env.n_alive()
    # the same steps under continuous load: up to SUSTAIN_STEPS untimed steps first (no rest), as many as
    # the seeds still waiting allow (a step retires ~950 streamlines; running dry would empty the slots)
    seeds_left = n_seeds - int(env._batch.ctrl_host[6])
    k_sus = min(args.steps, 50)
    pre = min(SUSTAIN_STEPS, seeds_left // 1100 - k_sus)
    sustained_ms = sustained_units = None
    if pre >= 100:
        for _ in range(pre):
            runner.step()
        env.n_alive()
        s_before = env.streamline_steps()
        sv0, sv1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sv0.record(stream)
        for _ in range(k_sus):
            runner.step()
        sv1.record(stream)
        torch.cuda.synchronize(dev)
        sustained_ms = sv0.elapsed_time(sv1)
        env.n_alive()
        sustained_units = env.streamline_steps() - s_before
        if int(env._batch.ctrl_host[env._cur]) < N_ACTOR:      # ran dry after all: not a valid sample
            sustained_ms = sustained_units = None
    saturated = bool(actor.overflowed() or env.operand_saturated())
    time.sleep(0.03)          # let the last clock samples of this leg arrive
    sm_mhz = sampler.median_between(t_begin, t_end) if sampler is not None else None
    return alg, {'elapsed_ms': elapsed_ms, 'units': units, 'gpu_launches': gpu_launches, 'alive_end': alive_end,
                 'prof': prof, 'saturated': saturated, 'sm_mhz': sm_mhz,
                 'sustained_ms': sustained_ms, 'sustained_units': sustained_units, 'outputs': outputs}


def run_e2e(env, alg, dev, world, barrier):
    """Public API, host buffers: pinned-host seeds H2D, full episodes incl. the low-occupancy tail, packed
    streamlines + flags back in host memory -- on rank 0 for every rank's share when N > 1 (the NCCL
    gather, the path's only collective, is inside the timed region)."""
    import torch
    from tracktolearn_b200.tracking.tracker import Tracker
    stream = torch.cuda.current_stream(dev)
    tracker = Tracker(alg, N_ACTOR, min_length=10.0, max_length=MAX_LENGTH_MM)
    # one untimed pass first: device buffers, pinned staging memory and NCCL's point-to-point channels are
    # set up once per process (the W >= 3 warm-up rule applies to this leg too), then the same call is timed
    for _ in tracker.track_gathered(env, copy=False):
        pass
    barrier()
    time.sleep(REST_S)      # a tracking job starts on an idle GPU, not on the heels of another 270 ms of full load
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    d2h = units = steps = n_streamlines = 0
    for batch in tracker.track_gathered(env, copy=False):
        units += env.streamline_steps()
        steps += alg.last_episode_steps
        if batch is not None:
            d2h += batch.data.nbytes + batch.offsets.nbytes + batch.data_per_streamline['flags'].nbytes
            n_streamlines += len(batch)
    e1.record(stream)
    barrier()
    return {'ms': e0.elapsed_time(e1), 'units': units, 'steps': steps, 'd2h': d2h, 'streamlines': n_streamlines,
            'h2d': len(env.seeds) * 3 * 8}


def run_sharded(args, dev, world, rank, actor_sd, prec, barrier):
    """BASELINE.json configs[2]: 290^3 0.5 mm volume, exactly 1 000 000 seeds -- one list, shuffled once
    (tracker.py:94), sharded in contiguous slices -- tracked by the streaming tracker on every GPU and
    gathered on rank 0.  Strong scaling: the total is fixed."""
    import torch
    import torch.distributed as dist
    from tracktolearn_b200 import parallel
    from tracktolearn_b200.algorithms.sac_auto import SACAuto
    from tracktolearn_b200.environments.utils import random_seeds_from_mask
    from tracktolearn_b200.tracking.tracker import Tracker
    t_setup = time.perf_counter()
    env, sub = make_env(SHARDED_SHAPE, SHARDED_VOXEL_MM, dev)
    seed_mask = sub['seed_mask'].cpu().numpy()
    del sub
    torch.cuda.empty_cache()
    rs = np.random.RandomState(1337)
    npv = max(1, -(-SHARDED_SEEDS // int(seed_mask.astype(bool).sum())))
    seeds = random_seeds_from_mask(seed_mask, npv, rs)
    rs.shuffle(seeds)
    seeds = seeds[:SHARDED_SEEDS]
    env.seeds = parallel.shard_seeds(seeds, rank, world)
    alg = SACAuto(STATE_SIZE, 3, HIDDEN, n_actors=N_ACTOR, device=dev, precision=prec)
    alg.agent.actor.load_state_dict(actor_sd)
    tracker = Tracker(alg, N_ACTOR, min_length=10.0, max_length=MAX_LENGTH_MM)
    stream = torch.cuda.current_stream(dev)
    setup_s = time.perf_counter() - t_setup
    for _ in tracker.track_gathered(env, copy=False):      # untimed: allocations, NCCL channels
        pass
    barrier()
    time.sleep(REST_S)
    barrier()
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    e0.record(stream)
    units = steps = 0
    merged = None
    for start, end, slots in tracker._passes(env):
        tracker._run_pass(env, start, end, slots)
        units += env.streamline_steps()
        steps += alg.last_episode_steps
        e1.record(stream)
        merged = parallel.gather_env_streamlines(env, copy=False)
    e2.record(stream)
    barrier()
    total_ms, track_ms = e0.elapsed_time(e2), e0.elapsed_time(e1)
    ok = True
    n_total = None
    if rank == 0:
        n_total = len(merged)
        lens = np.diff(merged.offsets)
        ok = bool(n_total == SHARDED_SEEDS and np.array_equal(merged.data_per_streamline['seeds'], seeds)
                  and np.array_equal(merged.data[merged.offsets[:-1]], seeds.astype(np.float32))
                  and lens.min() >= 1 and lens.max() <= env.max_nb_steps + 1
                  and (merged.data_per_streamline['flags'] != 0).all())
    t = torch.tensor([total_ms, track_ms, float(steps)], dtype=torch.float64, device=dev)
    u = torch.tensor([float(units)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(u, op=dist.ReduceOp.SUM)
    total_ms, track_ms, max_steps = float(t[0]), float(t[1]), float(t[2])
    occupancy = float(u[0]) / max(1.0, world * max_steps * N_ACTOR)
    return {
        'scaling': 'strong', 'metric': 'streamline-steps/sec', 'value': float(u[0]) / (total_ms * 1e-3),
        'unit': 'streamline-steps/s', 'precision': prec,
        'workload': '0.5mm-iso synthetic 290x290x290 order-8 fODF (auto step 0.375mm), %d seeds, one common '
                    'shuffle, sharded over %d GPU(s), n_actor %d per GPU' % (SHARDED_SEEDS, world, N_ACTOR),
        'total_ms': total_ms, 'tracking_ms_max_over_ranks': track_ms, 'gather_ms': total_ms - track_ms,
        'streamline_steps': float(u[0]), 'env_steps_max_over_ranks': max_steps,
        'mean_slot_occupancy': occupancy, 'streamlines_per_s': SHARDED_SEEDS / (total_ms * 1e-3),
        'limiter': ('mean slot occupancy %.2f: the longest streamline of a shard, not the GPU count, sets the number '
                    'of steps, and the steps after the seeds run out are latency-bound' % occupancy),
        'what': 'seeds H2D, streaming episodes incl. tail, device-side pack, NCCL gather of points / lengths / '
                'seeds / flags on rank 0, one D2H there; CUDA events, max over ranks',
        'gathered_streamlines': n_total, 'properties_ok': ok, 'setup_s': setup_s}


def main_gpu(args):
    quiet_stdout()
    import torch
    import torch.distributed as dist
    from tracktolearn_b200 import _lib, synthetic

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    lib = _lib.load()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---- workload: configs[1] ----------------------------------------------------------
    env, sub = make_env(SHAPE, VOXEL_MM, dev)
    seed_mask_np = sub['seed_mask'].cpu().numpy()
    env.seeds = sharded_seed_list(seed_mask_np, world, rank)
    seeds_all = env.seeds
    n_seeds = len(env.seeds)
    actor_sd = synthetic.actor_state_dict(STATE_SIZE, HIDDEN, seed=1111, kind='tracking')
    pk = peaks()
    traffic = ncu_traffic()

    # ---- device-resident throughput, every tier; the headline tier FIRST: this part is power-capped
    # (sw_power_cap is active through every leg) and a leg that follows 100+ ms of tensor-core load runs at
    # visibly lower SM clocks than the same leg on a rested chip (benchmarks/tier_repeat.py)
    main = args.precision
    order = [main] + [p for p in TIERS if p != main]
    if args.only_main:
        order = [main]
    # the clock sampler starts before the untimed steps: nvidia-smi needs 0.1-0.3 s before its first
    # sample, longer than a short timed region; only the samples taken between the two marks count
    sampler = ClockSampler(local_rank)
    sampler.start()
    results, alg_main = {}, None
    for prec in order:
        alg, r = run_tier(env, actor_sd, prec, args, dev, lib, barrier, sampler, prec == main)
        results[prec] = r
        if prec == main:
            alg_main = alg
        else:
            del alg
    clocks = sampler.stop()

    # ---- end to end through the public API, host buffers --------------------------------------
    e2e = None
    if not args.no_e2e:
        env.seeds = seeds_all[:min(n_seeds, E2E_SEEDS)]
        e2e = run_e2e(env, alg_main, dev, world, barrier)
        env.seeds = seeds_all

    # the TF32 denominator is measured AFTER the timed legs: ten 8192^3 cuBLAS products right before the
    # headline leg would hand it a chip that is already power-capped
    tf32_peak = measure_tf32_peak(dev)

    # ---- reduce over ranks: max time, summed units -------------------------------------------
    def reduce(ms, units):
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        u = torch.tensor([units], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(u, op=dist.ReduceOp.SUM)
        return float(t[0]), float(u[0])

    tiers = {}
    for prec in order:
        r = results[prec]
        ms, units_all = reduce(r['elapsed_ms'], r['units'])
        kernels = {name: {'launches': n, 'avg_us': 1000.0 * t_ms / n} for name, (n, t_ms) in sorted(r['prof'].items())}
        tiers[prec] = {'value': units_all / (ms * 1e-3), 'unit': 'streamline-steps/s', 'ms_per_step': ms / args.steps,
                       'tolerance': TIER_NOTE[prec], 'roofline': roofline_of(prec, r['prof'], r['alive_end'], pk,
                                                                              tf32_peak, traffic),
                       'kernels': kernels, 'saturated': r['saturated'], 'sm_mhz_timed_region': r['sm_mhz'],
                       'regime': 'rested chip: %d burn-in steps, %.1f s idle, W warm-up steps, K timed steps'
                                 % (BURN_IN, REST_S)}
        # every rank takes the same decision (same seeds per rank +-1, same step counts)
        s_ms, s_units = reduce(r['sustained_ms'] or 0.0, r['sustained_units'] or 0)
        tiers[prec]['sustained'] = None if not r['sustained_ms'] else {
            'value': s_units / (s_ms * 1e-3), 'unit': 'streamline-steps/s',
            'what': 'the same tier timed over min(K, 50) steps after ~125 ms of continuous load (no rest): '
                    'what sw_power_cap leaves of the rested-chip figure'}
    e2e_out = None
    if e2e is not None:
        ms, units_all = reduce(e2e['ms'], e2e['units'])
        e2e_out = {'value': units_all / (ms * 1e-3), 'unit': 'streamline-steps/s',
                   'h2d_bytes_per_step': e2e['h2d'] / max(1, e2e['steps']),
                   'd2h_bytes_per_step': e2e['d2h'] / max(1, e2e['steps']), 'precision': main, 'ms': ms,
                   'what': 'Tracker.track_gathered over %d seeds per GPU (one list, one common shuffle, sharded): '
                           'pinned-host seeds H2D, full episodes incl. tail, device-side pack, %s packed '
                           'streamlines+flags D2H on rank 0; %d env steps, %d streamlines on rank 0'
                           % (min(n_seeds, E2E_SEEDS), 'gather on rank 0 (shared pinned host arena, NCCL carries sizes and the barrier; NCCL point-to-point when the arena is unavailable), ' if world > 1 else '',
                              e2e['steps'], e2e['streamlines'])}

    # ---- HBM side of the two env kernels (main tier) ---------------------------------------------
    mr = results[main]
    prof, rows_prof = mr['prof'], mr['alive_end']

    def avg_ms(name):
        n, ms = prof.get(name, (0, 0.0))
        return ms / n if n else None
    op_bytes = 640 * (4 if main == 'tf32' else 2)
    # algorithmic bytes per row (SURVEY 8(d)); without the fp32 API tensor the state write is the operand
    # row instead of the 2460-byte fp32 row, and the direction history is the previous row's direction block
    # shifted by one direction instead of 100 fp32 points re-read (DESIGN.md section 4)
    state_write = op_bytes if args.operand_only else 2460 + 1280
    dirs_read = (300 * op_bytes // 640) if args.operand_only else 1200
    state_bytes = 4680 + state_write + dirs_read + 12
    step_bytes = 4680 + state_write + dirs_read + 512 + 48
    state_ms = avg_ms('build_state_kernel')
    step_ms = sum(avg_ms(k) or 0.0 for k in ('propagate_stop_kernel', 'build_state_kernel'))
    roofline_step = None
    if state_ms and step_ms:
        a_state = state_bytes * rows_prof / (state_ms * 1e-3) / 1e9
        a_step = step_bytes * rows_prof / (step_ms * 1e-3) / 1e9
        roofline_step = {
            'build_state_kernel': {'bound': 'hbm', 'achieved': a_state, 'peak': pk['hbm_gbs'], 'unit': 'GB/s',
                                   'frac': a_state / pk['hbm_gbs'], 'traffic': traffic.get('build_state_kernel'),
                                   'algorithmic_bytes_per_launch': state_bytes * rows_prof,
                                   'bytes_per_row': state_bytes},
            'env_step (propagate_stop+build_state)': {
                'bound': 'hbm', 'achieved': a_step, 'peak': pk['hbm_gbs'], 'unit': 'GB/s',
                'frac': a_step / pk['hbm_gbs'],
                'traffic': (traffic.get('build_state_kernel', 0) + traffic.get('propagate_stop_kernel', 0)) or None,
                'algorithmic_bytes_per_launch': step_bytes * rows_prof, 'bytes_per_row': step_bytes},
            'note': 'algorithmic bytes over kernel time: an effective rate.  The DRAM traffic ncu sees is a fraction '
                    'of it (neighbouring rows share voxels in L1/L2); the state kernel is bound by the L1 data pipe '
                    'and gather latency, not by DRAM (DESIGN.md section 4)',
            'peak_source': pk['source']}

    # ---- configs[2], sharded (strong scaling) -----------------------------------------------------
    sharded = None
    if not args.no_sharded:
        del alg_main
        env._batch = None
        torch.cuda.empty_cache()
        sharded = run_sharded(args, dev, world, rank, actor_sd, main, barrier)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu:
        sub_np = {'sh': sub['sh'].cpu().numpy(), 'mask': sub['mask'].cpu().numpy()}
        res, choice = cpu_reference_best(sub_np, seeds_all, actor_sd, 5, 1, probe_steps=2)
        cpu_baseline = {'value': res['value'], 'unit': 'streamline-steps/s', 'cores': os.cpu_count() or 1,
                        'kind': 'port',
                        'sample': '5 act->step->harvest iterations (after 1 warm-up) over the same %d-streamline batch '
                                  'of the same volume and seeds; numpy/scipy env restatement + torch-CPU fp32 actor; '
                                  'scipy map_coordinates is single-threaded' % N_ACTOR,
                        'ms_per_step': res['ms_per_step'], 'threads': choice, 'phase_seconds': res['phase_s']}

    if rank == 0:
        t = tiers[main]
        line = {
            'metric': 'streamline-steps/sec', 'value': t['value'], 'unit': 'streamline-steps/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': t['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': main, 'data': 'synthetic',
            'config': workload_config(),
            'run': {'headline_tier': main, 'seeds_per_gpu': n_seeds,
                    'seeds': 'one list (npv=20 per GPU over the mask shell), one common shuffle, contiguous shards',
                    'streaming_refill': True,
                    'slot_order': 'seeds enter the slots in voxel raster order (rows / output keep the shuffled order)'
                    if os.environ.get('TTL_LOCALITY', '1') != '0' else 'row (shuffled) order',
                    'launch': 'programmatic dependent launch' if os.environ.get('TTL_PDL', '1') != '0' else 'plain',
                    'alive_at_end': mr['alive_end'], 'burn_in_steps': BURN_IN,
                    'state_rows': ('actor operand rows only; the fp32 API tensor is not materialised in the '
                                   'device loop (SURVEY 7 step 7)' if args.operand_only
                                   else 'fp32 API tensor + actor operand rows'),
                    'l2': 'inputs larger than L2: %d MB SH volume + 2x64 MB operand rows + 205 MB activations'
                          % (SHAPE[0] * SHAPE[1] * SHAPE[2] * 48 * 4 // 1000000),
                    'parallelism': 'seeds sharded, volume replicated, no data-path collective; NCCL only for the '
                                   'final tractogram gather (inside e2e and sharded)',
                    'tf32_peak_tflops_measured': tf32_peak},
            'e2e': e2e_out,
            'gpu_launches': mr['gpu_launches'],
            'clocks': clocks,
            'roofline': t['roofline'],
            'roofline_step_kernels': roofline_step,
            'kernels': t['kernels'],
            'sustained': tiers[main].get('sustained'),
            'tiers': tiers,
            'sharded': sharded,
            'cpu_baseline': cpu_baseline,
            'flop_per_streamline_step': ACTOR_FLOP_PER_ROW,
        }
        if args.dump_outputs:
            write_outputs(args.dump_outputs, mr['outputs'])
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--precision', default='fp16', choices=list(TIERS),
                    help='headline tier (value / e2e / sharded / roofline); the others are reported under `tiers`')
    ap.add_argument('--only-main', action='store_true', help='skip the other tiers (profiling runs)')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--fp32-state', dest='operand_only', action='store_false',
                    help='also materialise the fp32 state rows every step (the reference API tensor)')
    ap.add_argument('--graph', action='store_true', help='replay the kernels of a step from a CUDA graph')
    ap.add_argument('--no-e2e', action='store_true', help='skip the end-to-end leg (profiling runs)')
    ap.add_argument('--no-sharded', action='store_true', help='skip the configs[2] sharded leg')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="write the headline tier's outputs after its last timed step as DIR/<name>.npy")
    ap.add_argument('--cpu-worker', default=None, help=argparse.SUPPRESS)
    ap.add_argument('--torch-threads', type=int, default=os.cpu_count() or 1, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.cpu_worker:
        sys.exit(cpu_worker(a))
    if a.dump_outputs and a.impl == 'reference':
        ap.error('--dump-outputs dumps the GPU step path; the reference arm has no such output')
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.warmup < 3:
        a.warmup = 3
    sys.exit(main_reference(a) if a.impl == 'reference' else main_gpu(a))
