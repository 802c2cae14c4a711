"""bench.py --impl reference (the CPU arm beside the GPU arm) prints one JSON line with the benchmark's keys; runs without a
GPU (one step over the whole C2 batch with the oracle: ~20 s).  On the GPU, --dump-outputs writes the last timed step's
outputs, which match the oracle on the same seeded inputs."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, str(ROOT / 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0'],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert key in d, key
    assert d['impl'] == 'reference' and d['metric'] == 'mel_frames_per_sec_fwd' and d['unit'] == 'frames/s'
    assert d['higher_is_better'] is True and d['steps'] == 1 and d['value'] > 0
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert d['config']['workload'].startswith('C2: LJ256 ForwardTransformer inference')


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_step(tmp_path):
    from oracle import forward_oracle as fo
    out = tmp_path / 'out'
    r = subprocess.run([sys.executable, str(ROOT / 'bench.py'), '--steps', '2', '--warmup', '1', '--no-cpu-baseline', '--no-train',
                        '--dump-outputs', str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith('{')][-1])
    assert d['steps'] == 2
    files = {f.stem: np.load(f) for f in out.glob('*.npy')}
    assert set(files) == {'mel', 'duration', 'pitch', 'expanded_mask', 'int_durations', 'mel_lengths'}
    assert all(a.dtype in (np.float32, np.float64) for a in files.values())
    assert sum(a.nbytes for a in files.values()) <= 64 << 20
    assert files['mel'].shape == (64, 1000, 80)
    # the first row of the seeded batch against the oracle (bench.py: weights seed 7, inputs seed 200 on rank 0)
    cfg = fo.CONFIGS['LJ256']
    tok, dur, pit = fo.make_inputs('full', 64, 128, 1000, seed=200)
    with torch.no_grad():
        ref = fo.forward_transformer_call(fo.init_params(cfg, seed=7), cfg, tok[:1], dur[:1, :, None], pit[:1, :, None])
    n = ref['mel'].shape[1]
    assert np.array_equal(files['int_durations'][0], dur[0].numpy())
    assert float(np.abs(files['mel'][0, :n] - ref['mel'][0].numpy()).max()) < 1e-3
