"""The reference arm of bench.py runs on CPU: check the one-JSON-line contract the round driver parses (no GPU needed)."""
import json, os, subprocess, sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line(tmp_path):
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE='1')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '1',
                          '--dump-outputs', str(tmp_path / 'dump')],
                         capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines                                   # stdout carries the JSON line and nothing else
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['metric'] == 'rgbd_pair_frames_per_sec' and d['unit'] == 'pairs/s'
    assert d['higher_is_better'] is True and d['n_gpus'] == 1 and d['steps'] == 1 and d['value'] > 0
    assert d['cpu_baseline']['kind'] in ('port', 'reference') and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    # same config as the GPU arm: the full 64-pair step and the very same workload string (the driver compares them)
    sys.path.insert(0, ROOT)
    import bench
    assert d['config']['workload'] == bench.workload_string(64) and d['config']['tracks_per_gpu'] == 64
    assert 'all 64 pairs' in d['cpu_baseline']['sample']
    # --dump-outputs: the last timed step's poses, one 4x4 per pair of the workload
    assert os.listdir(str(tmp_path / 'dump')) == ['poses.npy']
    poses = np.load(str(tmp_path / 'dump' / 'poses.npy'))
    assert poses.shape == (64, 4, 4) and poses.dtype == np.float64 and np.isfinite(poses).all()
    assert np.array_equal(poses[:, 3], np.tile([0.0, 0.0, 0.0, 1.0], (64, 1)))


def test_steps_must_be_positive():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '0'],
                         capture_output=True, text=True, timeout=300, env=dict(os.environ, PYTHONDONTWRITEBYTECODE='1'), cwd=ROOT)
    assert out.returncode == 2 and '--steps' in out.stderr and out.stdout == ''


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE='1', RANK='1', WORLD_SIZE='2', LOCAL_RANK='1')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2', '--steps', '1', '--warmup', '1'],
                         capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert out.returncode == 0 and out.stdout.strip() == ''
