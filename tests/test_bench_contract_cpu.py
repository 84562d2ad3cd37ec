"""bench.py's JSON contract, checked on the CPU (reference arm) with the smallest configuration."""
import json
import os
import subprocess
import sys

import numpy as np

from conftest import ROOT


def _run(*args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + list(args), stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, universal_newlines=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1, r.stdout
    return json.loads(lines[0])


def test_reference_arm_line():
    j = _run('--impl', 'reference', '--config', 'cfg1', '--steps', '2', '--warmup', '1')
    assert j['impl'] == 'reference' and j['metric'] == 'RRI sweeps/sec' and j['unit'] == 'sweeps/s'
    assert j['higher_is_better'] is True and j['n_gpus'] == 1 and j['steps'] == 2 and j['warmup'] == 1
    assert j['value'] > 0 and abs(j['ms_per_step'] * j['value'] - 1e3) < 1e-6 * 1e3
    assert j['vs_baseline'] is None and j['data'] == 'synthetic' and 'workload' in j['config']
    cb = j['cpu_baseline']
    assert cb['kind'] in ('port', 'reference') and cb['value'] == j['value'] and 'sample' in cb
    # all host cores, whatever OMP_NUM_THREADS says (torch.distributed.run exports OMP_NUM_THREADS=1)
    assert cb['cores'] == len(os.sched_getaffinity(0)) == cb['host_cores']
    assert j['e2e'] == {'value': j['value'], 'unit': 'sweeps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def test_reference_arm_full_threads_under_torchrun_env():
    """rank 0 of a torchrun launch: OMP_NUM_THREADS=1 in the environment must not reduce the CPU arm to one thread;
    RRI_BENCH_PORT=1 selects the NumPy port even when the reference copy is present"""
    env = dict(os.environ, RANK='0', WORLD_SIZE='2', LOCAL_RANK='0', OMP_NUM_THREADS='1', RRI_BENCH_PORT='1')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2',
                        '--config', 'cfg1', '--steps', '1', '--warmup', '0'], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, universal_newlines=True, timeout=120)
    assert r.returncode == 0, r.stderr[-2000:]
    j = json.loads([l for l in r.stdout.splitlines() if l.startswith('{')][0])
    assert j['cpu_baseline']['cores'] == len(os.sched_getaffinity(0)) and j['cpu_baseline']['kind'] == 'port'


def test_reference_arm_dump_outputs(tmp_path):
    """--dump-outputs: W and T after the last timed sweep, the same from run to run; --steps sets how many sweeps"""
    args = ('--impl', 'reference', '--config', 'cfg1', '--warmup', '1', '--dump-outputs')
    for name, steps in (('a', '2'), ('b', '2'), ('c', '3')):
        _run('--steps', steps, *(args + (str(tmp_path / name),)))

    def ld(run, f):
        return np.load(str(tmp_path / run / f))
    W, T = ld('a', 'W.npy'), ld('a', 'T.npy')
    assert W.shape == (500, 10) and T.shape == (10, 300) and W.dtype == T.dtype == np.float64
    assert np.allclose(W, ld('b', 'W.npy'), rtol=1e-12, atol=0) and np.allclose(T, ld('b', 'T.npy'), rtol=1e-12, atol=0)
    assert not np.allclose(W, ld('c', 'W.npy'))


def test_dump_outputs_samples_rows_beyond_the_cap(tmp_path):
    import bench
    n, k = 150000, 64
    W = np.random.RandomState(1).rand(n, k)
    W[:, 0] = np.arange(n)
    T = np.random.RandomState(2).rand(k, 2000)
    for name in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / name), n, 0, W, T)
    files = [str(tmp_path / 'a' / f) for f in ('W.npy', 'T.npy')]
    assert sum(os.path.getsize(f) for f in files) <= bench.DUMP_BYTES
    Ws = np.load(files[0])
    rows = Ws[:, 0].astype(np.int64)
    assert 0 < len(rows) < n and np.all(np.diff(rows) > 0) and np.array_equal(Ws, W[rows])
    assert np.array_equal(Ws, np.load(str(tmp_path / 'b' / 'W.npy')))
    assert np.array_equal(np.load(files[1]), T)
    # a T larger than the cap by itself: a sample of its columns, and W still fits next to it
    T = np.random.RandomState(3).rand(k, 200000)
    T[0] = np.arange(T.shape[1])
    bench.dump_outputs(str(tmp_path / 'c'), 1000, 0, W[:1000], T)
    files = [str(tmp_path / 'c' / f) for f in ('W.npy', 'T.npy')]
    assert sum(os.path.getsize(f) for f in files) <= bench.DUMP_BYTES
    Ts = np.load(files[1])
    cols = Ts[0].astype(np.int64)
    assert 0 < len(cols) < T.shape[1] and np.all(np.diff(cols) > 0) and np.array_equal(Ts, T[:, cols])
    assert np.array_equal(np.load(files[0]), W[:1000])


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2', LOCAL_RANK='1')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2',
                        '--config', 'cfg1', '--steps', '1', '--warmup', '0'], env=env, stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, universal_newlines=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ''
