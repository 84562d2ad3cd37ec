"""bench.py --dump-outputs on the device paths: the files hold exactly what the timed sweeps computed."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, relfro

pytestmark = pytest.mark.gpu

ROWS = 16384


def _bench(out, *args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--rows', str(ROWS), '--no-e2e', '--no-cpu',
                        '--no-rri', '--dump-outputs', str(out)] + list(args), stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, universal_newlines=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return np.load(str(out / 'W.npy')), np.load(str(out / 'T.npy'))


def test_dump_is_the_engine_result_after_warmup_plus_steps(cuda_device, tmp_path):
    import bench
    import rri_nmf_b200 as R
    W2, T2 = _bench(tmp_path / 'a', '--steps', '2', '--warmup', '1')
    W3, _ = _bench(tmp_path / 'b', '--steps', '3', '--warmup', '1')
    assert W2.shape == (ROWS, 64) and T2.shape == (64, 20000) and W2.dtype == T2.dtype == np.float32
    assert not np.array_equal(W2, W3)
    X, W0, T0 = bench.gen_shard(torch, bench.CONFIGS['cfg3'], ROWS, 0, cuda_device)
    eng = R.RRIEngine(X, 64, order='hals', math='tf32')
    W, T = W0.clone(), T0.clone()
    eng.sweeps(W, T, 3, eng.params())                # 1 warm-up + 2 timed sweeps, bit for bit (test_gpu_fullsize)
    assert np.array_equal(W.cpu().numpy(), W2) and np.array_equal(T.cpu().numpy(), T2)
    eng.close()


@pytest.mark.parametrize('masked', ['dense', 'sparse'])
def test_dump_of_the_masked_config(cuda_device, tmp_path, masked):
    import bench
    import rri_nmf_b200 as R
    Wd, Td = _bench(tmp_path, '--config', 'cfg4', '--masked', masked, '--steps', '1', '--warmup', '0')
    assert Wd.shape == (ROWS, 50) and Td.shape == (50, 20000) and Wd.dtype == Td.dtype == np.float32
    cfg = bench.CONFIGS['cfg4']
    X, W0, T0 = bench.gen_shard(torch, cfg, ROWS, 0, cuda_device)
    M = bench.gen_mask_shard(torch, cfg, ROWS, 0, cuda_device)
    if masked == 'sparse':
        eng = R.RRIEngine((X * M).to_sparse_csr(), 50, order='rri')
    else:
        eng = R.RRIEngine(X, 50, W_mat=M, order='rri', math='tf32')
    W, T = W0.clone(), T0.clone()
    eng.sweeps(W, T, 1, eng.params(ub_t=1.0))
    assert relfro(Wd, W.cpu().numpy()) < 1e-6 and relfro(Td, T.cpu().numpy()) < 1e-6
    assert relfro(Wd, W0.cpu().numpy()) > 1e-2
    eng.close()
