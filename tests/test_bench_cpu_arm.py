"""bench.py's CPU legs: the reference arm must be the UNMODIFIED reference whenever it is importable
(installed under baseline/_ref), the oracle port otherwise."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from tapnet_b200 import synth  # noqa: E402


def test_cpu_arm_runs_the_unmodified_reference_when_importable():
  have_ref = os.path.isfile(os.path.join(ROOT, 'baseline', '_ref', 'tapnet', 'torch', 'tapir_model.py'))
  wl = dict(bench.WORKLOADS['c2'], frames=6)
  video = synth.make_video(6)
  queries = synth.make_queries(32, 6)
  arm = bench.CpuArm(synth.make_state_dict(0), video, queries, wl)
  assert arm.kind == ('reference' if have_ref else 'port')
  if have_ref:
    assert type(arm.model).__module__ == 'tapnet.torch.tapir_model'
  torch.set_num_threads(min(8, os.cpu_count() or 1))
  arm.threads, arm.sweep = torch.get_num_threads(), {}
  sec = arm.sample()
  d = arm.describe(sec)
  assert sec > 0 and d['kind'] == arm.kind and d['unit'] == bench.UNIT
  assert abs(d['value'] - 32 * 6 / sec) < 1e-6 * d['value'] + 0.1


def test_dump_outputs_writes_float32_and_samples_queries_above_the_limit(tmp_path, monkeypatch):
  import numpy as np
  N, T = 40, 6
  g = torch.Generator().manual_seed(0)
  out = dict(tracks=torch.randn(1, N, T, 2, generator=g), occlusion=torch.randn(1, N, T, generator=g),
             unrefined_tracks=[torch.randn(1, N, T, 2, generator=g) for _ in range(3)])
  bench.dump_outputs(str(tmp_path / 'all'), out, N, 1, 0)
  got = {k: np.load(tmp_path / 'all' / f'{k}.npy') for k in out}
  assert sorted(os.listdir(tmp_path / 'all')) == sorted(f'{k}.npy' for k in out)
  assert all(a.dtype == np.float32 for a in got.values())
  np.testing.assert_array_equal(got['tracks'], out['tracks'].numpy())
  np.testing.assert_array_equal(got['unrefined_tracks'], torch.stack(out['unrefined_tracks']).numpy())
  limit = 4096
  monkeypatch.setattr(bench, 'DUMP_LIMIT', limit)
  for run in ('a', 'b'):
    bench.dump_outputs(str(tmp_path / run), out, N, 1, 0)
  files = sorted(os.listdir(tmp_path / 'a'))
  assert files == sorted(os.listdir(tmp_path / 'b')) and 'query_index.npy' in files
  assert sum(os.path.getsize(tmp_path / 'a' / f) - 128 for f in files) <= limit  # 128 B .npy header
  idx = np.load(tmp_path / 'a' / 'query_index.npy').astype(np.int64)
  assert 0 < len(idx) < N and np.all(np.diff(idx) > 0)
  for f in files:
    np.testing.assert_array_equal(np.load(tmp_path / 'a' / f), np.load(tmp_path / 'b' / f))
  np.testing.assert_array_equal(np.load(tmp_path / 'a' / 'tracks.npy'), got['tracks'][:, idx])
  np.testing.assert_array_equal(np.load(tmp_path / 'a' / 'unrefined_tracks.npy'),
                                got['unrefined_tracks'][:, :, idx])


def _run_reference_arm(rank, world):
  import subprocess
  env = dict(os.environ, RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world),
             MASTER_ADDR='127.0.0.1', MASTER_PORT='29577')
  return subprocess.run(
      [sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', str(world),
       '--steps', '1', '--warmup', '0'], capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)


def test_reference_arm_line_and_rank_behaviour():
  """`bench.py --impl reference` as the driver launches it for N = 2: rank 0 alone works and prints
  ONE JSON line with the own-arm keys plus impl / cpu_baseline / e2e; the other ranks exit 0
  without output and without touching a GPU or the process group."""
  import json
  other = _run_reference_arm(1, 2)
  assert other.returncode == 0 and other.stdout.strip() == '', other.stderr[-2000:]
  first = _run_reference_arm(0, 2)
  assert first.returncode == 0, first.stderr[-2000:]
  lines = [l for l in first.stdout.splitlines() if l.startswith('{')]
  assert len(lines) == 1
  d = json.loads(lines[0])
  assert d['impl'] == 'reference' and d['n_gpus'] == 2 and d['unit'] == bench.UNIT
  assert d['higher_is_better'] is True and d['scaling'] == 'weak' and d['vs_baseline'] is None
  assert d['config']['queries'] == 2 * bench.WORKLOADS['c2']['q_per_gpu']
  assert d['cpu_baseline']['value'] == d['value'] == d['e2e']['value'] > 0
  assert d['cpu_baseline']['kind'] in ('reference', 'port') and d['cpu_baseline']['cores'] >= 1
  assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0
