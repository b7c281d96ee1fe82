"""bench.py contract.  Without a GPU: the `--impl reference` arm's JSON line (the oracle port on the host cores,
one 64x96-free full-size frame per step is too slow here, so the contract is checked on the smallest legal run) and
the stock-PyTorch context leg on the CPU device (same code path as on the GPU, minus the CUDA synchronisations).
With a GPU (-m gpu): `--steps` and `--dump-outputs` of the device path."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
  r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0'],
                     capture_output=True, text=True, timeout=600, cwd=ROOT)
  assert r.returncode == 0, r.stderr[-2000:]
  lines = [l for l in r.stdout.splitlines() if l.strip()]
  assert len(lines) == 1, r.stdout
  d = json.loads(lines[0])
  assert d['impl'] == 'reference' and d['unit'] == 'frames/s' and d['higher_is_better'] is True
  assert d['metric'] == 'frames/sec (device-timed) DLA-34 512x512'
  assert d['value'] > 0 and d['steps'] == 1
  assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
  assert d['e2e'] == {'value': d['value'], 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def test_stock_pytorch_context_leg_runs_on_the_cpu_device():
  sys.path.insert(0, ROOT)
  import bench
  from centertrack_b200 import synthetic as wt
  from helpers import make_model
  opt, model, sd = make_model('coco_tracking')
  saved = bench.K
  bench.K = 40
  try:
    r = bench.stock_pytorch_leg(sd, opt.heads, 2, 64, 96, torch.device('cpu'), wt, steps=1, warmup=0)
  finally:
    bench.K = saved
  assert r['kind'] == 'port' and r['fp32'] > 0 and r['bf16_autocast'] > 0 and r['frames_per_step'] == 2


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step_repeat_exactly(tmp_path):
  """--dump-outputs writes the records and track tables of the last timed step; the inputs are seeded, so two runs
  with the same arguments dump the same arrays.  --steps is the number of timed steps the line reports."""
  from centertrack_b200 import _lib as L
  dumps = []
  for run in range(2):
    out = tmp_path / str(run)
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', '4', '--warmup', '3',
                        '--batch', '2', '--no-cpu-baseline', '--no-parity', '--no-latency', '--no-gpu-baseline',
                        '--no-accurate', '--dump-outputs', str(out)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip())
    assert line['steps'] == 4
    assert sorted(os.listdir(str(out))) == ['records.npy', 'track_counts.npy', 'tracks.npy']
    d = {k: np.load(str(out / (k + '.npy'))) for k in ('records', 'tracks', 'track_counts')}
    assert d['records'].dtype == np.float32 and d['records'].shape[:2] == (2, 100)
    assert d['tracks'].dtype == np.float32 and d['tracks'].shape[0] == 2 and d['tracks'].shape[2] == L.CT_TRK_FLOATS
    assert d['track_counts'].dtype == np.float64 and d['track_counts'].shape == (2, 2)
    assert d['track_counts'][:, 0].sum() > 0 and d['records'][:, 0, 0].min() > 0
    dumps.append(d)
  for k in dumps[0]:
    assert np.array_equal(dumps[0][k], dumps[1][k]), k
