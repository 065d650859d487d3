"""bench.py --dump-outputs: what the last timed step computed, as one .npy file per array, so that two
builds of the project can be compared output for output on identical seeded inputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_writes_one_float_npy_per_array(tmp_path):
  bench.dump_outputs(str(tmp_path), {'loss/total': torch.tensor(1.5), 'indices': torch.arange(5),
                                     'param/core/kernel': torch.ones(3, 4), 'norm': torch.tensor(2.0, dtype=torch.float64)})
  assert sorted(os.listdir(tmp_path)) == ['indices.npy', 'loss.total.npy', 'norm.npy', 'param.core.kernel.npy']
  idx = np.load(tmp_path / 'indices.npy')
  assert idx.dtype == np.float64 and idx.tolist() == [0, 1, 2, 3, 4]
  k = np.load(tmp_path / 'param.core.kernel.npy')
  assert k.dtype == np.float32 and k.shape == (3, 4)
  assert np.load(tmp_path / 'loss.total.npy') == np.float32(1.5)
  assert np.load(tmp_path / 'norm.npy').dtype == np.float64


def test_dump_outputs_refuses_more_than_64_MB(tmp_path):
  with pytest.raises(SystemExit):
    bench.dump_outputs(str(tmp_path / 'out'), {'a': torch.zeros(8 << 20), 'b': torch.zeros((8 << 20) + 1)})
  assert not os.path.exists(tmp_path / 'out')


@pytest.mark.parametrize('argv', [['--steps', '0'], ['--impl', 'reference', '--dump-outputs', 'out']])
def test_bench_refuses_arguments_it_cannot_honour(argv):
  r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + argv, capture_output=True, text=True,
                     timeout=120)
  assert r.returncode == 2 and r.stdout == '', r.stderr[-2000:]


def _bench_dump(out):
  r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '2', '--warmup', '3', '--batch', '4',
                      '--unroll', '4', '--no-extras', '--dump-outputs', str(out)],
                     capture_output=True, text=True, timeout=600)
  assert r.returncode == 0, r.stderr[-2000:]
  line = json.loads(r.stdout)
  assert line['steps'] == 2
  return {f: np.load(os.path.join(out, f)) for f in sorted(os.listdir(out))}


@pytest.mark.gpu
def test_flagship_dump_is_identical_from_run_to_run(tmp_path):
  a, b = _bench_dump(tmp_path / 'a'), _bench_dump(tmp_path / 'b')
  assert a.keys() == b.keys()
  for name in ('loss.total.npy', 'param.policy_logits.kernel.npy', 'grad.policy_logits.kernel.npy',
               'param.entropy_cost_param.npy', 'grad.entropy_cost_param.npy'):
    assert name in a, sorted(a)
  assert sum(v.nbytes for v in a.values()) <= bench.DUMP_LIMIT_BYTES
  for name in a:
    assert a[name].dtype in (np.float32, np.float64), name
    assert np.all(np.isfinite(a[name])), name
    np.testing.assert_array_equal(a[name], b[name], err_msg=name)
  assert np.abs(a['grad.policy_logits.kernel.npy']).max() > 0
